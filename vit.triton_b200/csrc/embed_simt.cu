// Exact-fp32 / odd-shape helpers around the patch embedding:
//   patching        (B,C,H,W) -> (B, n, C*P*P) patch rows in (c, i, j) order.  Same contract as the
//                   reference's exported-but-unused `patching` entry point
//                   (vit/kernels/patching.py:54-92, torch restatement :95-105).
//   embed_finalize  x[b,t,:] = prefix_rows[t] + pos[t] for t < prefix ; x[b,t,:] += pos[t]  (vit/vit.py:195-200);
//                   prefix_rows = [cls] (ViT) or [cls; distillation token] (DeiT)
//   conv2d_nchw     generic strided conv with stride == kernel (vit/kernels/conv2d.py:100-150),
//                   output (B, O, H/kh, W/kw) like the reference; used by the standalone entry point.
#include "common.cuh"

namespace vt {

namespace {

__device__ __forceinline__ float ldf(const float* p) { return *p; }
__device__ __forceinline__ float ldf(const __nv_bfloat16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void stf(float* p, float v) { *p = v; }
__device__ __forceinline__ void stf(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

template <typename T>
__global__ void patching_kernel(const T* __restrict__ img, T* __restrict__ out, int B, int C, int H,
                                int W, int P) {
  const int gw = W / P, gh = H / P;
  const long long K = static_cast<long long>(C) * P * P;
  const long long total = static_cast<long long>(B) * gh * gw * K;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int k = static_cast<int>(idx % K);
  const long long pr = idx / K;
  const int patch = static_cast<int>(pr % (gh * gw));
  const int b = static_cast<int>(pr / (gh * gw));
  const int c = k / (P * P);
  const int rem = k - c * P * P;
  const int i = rem / P, j = rem - i * P;
  const int py = patch / gw, px = patch - py * gw;
  out[idx] = img[((static_cast<long long>(b) * C + c) * H + (py * P + i)) * W + px * P + j];
}

template <typename T>
__global__ void embed_finalize_kernel(T* __restrict__ x, const T* __restrict__ pos,
                                      const T* __restrict__ prefix_rows, int B, int N, int D, int prefix) {
  const long long total = static_cast<long long>(B) * N * D;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int d = static_cast<int>(idx % D);
  const int t = static_cast<int>((idx / D) % N);
  const float pv = ldf(pos + static_cast<long long>(t) * D + d);
  const float v = (t < prefix) ? ldf(prefix_rows + static_cast<long long>(t) * D + d) : ldf(x + idx);
  stf(x + idx, v + pv);
}

// embed_finalize with bool_masked_pos: a masked patch's projection is replaced by the mask token before pos is added
template <typename T>
__global__ void embed_finalize_masked_kernel(T* __restrict__ x, const T* __restrict__ pos,
                                             const T* __restrict__ prefix_rows, const T* __restrict__ mask_token,
                                             const uint8_t* __restrict__ mask, int B, int N, int D, int prefix) {
  const long long total = static_cast<long long>(B) * N * D;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int d = static_cast<int>(idx % D);
  const long long bt = idx / D;
  const int t = static_cast<int>(bt % N);
  const long long b = bt / N;
  const float pv = ldf(pos + static_cast<long long>(t) * D + d);
  float v;
  if (t < prefix) v = ldf(prefix_rows + static_cast<long long>(t) * D + d);
  else if (mask[b * (N - prefix) + t - prefix]) v = ldf(mask_token + d);
  else v = ldf(x + idx);
  stf(x + idx, v + pv);
}

// One thread per output element; weights are read with k fastest within a thread so consecutive
// output channels do not coalesce — this entry point exists for API parity, the model path uses
// vt_patch_embed_gemm (bf16) or patching + a GEMM (fp32).
template <typename T>
__global__ void conv2d_nchw_kernel(const T* __restrict__ in, const T* __restrict__ w,
                                   const T* __restrict__ bias, T* __restrict__ out, int B, int C,
                                   int H, int W, int O, int kh, int kw) {
  const int oh = H / kh, ow = W / kw;
  const long long total = static_cast<long long>(B) * O * oh * ow;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int x = static_cast<int>(idx % ow);
  const int y = static_cast<int>((idx / ow) % oh);
  const int o = static_cast<int>((idx / (static_cast<long long>(ow) * oh)) % O);
  const int b = static_cast<int>(idx / (static_cast<long long>(ow) * oh * O));
  float acc = 0.f;
  for (int c = 0; c < C; ++c)
    for (int i = 0; i < kh; ++i) {
      const T* ip = in + ((static_cast<long long>(b) * C + c) * H + (y * kh + i)) * W + x * kw;
      const T* wp = w + ((static_cast<long long>(o) * C + c) * kh + i) * kw;
      for (int j = 0; j < kw; ++j) acc = fmaf(ldf(ip + j), ldf(wp + j), acc);
    }
  stf(out + idx, acc + ldf(bias + o));
}

}  // namespace

int patching(const void* img, void* out, int B, int C, int H, int W, int P, int dtype,
             cudaStream_t stream) {
  if (!img || !out || B < 0 || C <= 0 || P <= 0 || H % P || W % P) return VT_ERR_ARG;
  const long long total = static_cast<long long>(B) * C * H * W;
  if (total == 0) return VT_OK;
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  if (dtype == VT_F32)
    patching_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(img),
                                                     static_cast<float*>(out), B, C, H, W, P);
  else if (dtype == VT_BF16)
    patching_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(
        static_cast<const __nv_bfloat16*>(img), static_cast<__nv_bfloat16*>(out), B, C, H, W, P);
  else
    return VT_ERR_DTYPE;
  return static_cast<int>(cudaGetLastError());
}

int embed_finalize(void* x, const void* pos, const void* prefix_rows, int B, int N, int D, int dtype, int prefix,
                   cudaStream_t stream) {
  if (!x || !pos || !prefix_rows || B < 0 || N < prefix || D <= 0 || prefix < 1 || prefix > 2) return VT_ERR_ARG;
  const long long total = static_cast<long long>(B) * N * D;
  if (total == 0) return VT_OK;
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  if (dtype == VT_F32)
    embed_finalize_kernel<float><<<grid, 256, 0, stream>>>(
        static_cast<float*>(x), static_cast<const float*>(pos), static_cast<const float*>(prefix_rows), B,
        N, D, prefix);
  else if (dtype == VT_BF16)
    embed_finalize_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(
        static_cast<__nv_bfloat16*>(x), static_cast<const __nv_bfloat16*>(pos),
        static_cast<const __nv_bfloat16*>(prefix_rows), B, N, D, prefix);
  else
    return VT_ERR_DTYPE;
  return static_cast<int>(cudaGetLastError());
}

int embed_finalize_masked(void* x, const void* pos, const void* prefix_rows, const void* mask_token, const void* mask,
                          int B, int N, int D, int dtype, int prefix, cudaStream_t stream) {
  if (!x || !pos || !prefix_rows || !mask_token || !mask || B < 0 || N < prefix || D <= 0 || prefix < 1 || prefix > 2)
    return VT_ERR_ARG;
  const long long total = static_cast<long long>(B) * N * D;
  if (total == 0) return VT_OK;
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  const uint8_t* m = static_cast<const uint8_t*>(mask);
  if (dtype == VT_F32)
    embed_finalize_masked_kernel<float><<<grid, 256, 0, stream>>>(
        static_cast<float*>(x), static_cast<const float*>(pos), static_cast<const float*>(prefix_rows),
        static_cast<const float*>(mask_token), m, B, N, D, prefix);
  else if (dtype == VT_BF16)
    embed_finalize_masked_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(
        static_cast<__nv_bfloat16*>(x), static_cast<const __nv_bfloat16*>(pos),
        static_cast<const __nv_bfloat16*>(prefix_rows), static_cast<const __nv_bfloat16*>(mask_token), m, B, N, D,
        prefix);
  else
    return VT_ERR_DTYPE;
  return static_cast<int>(cudaGetLastError());
}

int conv2d_nchw(const void* in, const void* w, const void* bias, void* out, int B, int C, int H,
                int W, int O, int kh, int kw, int dtype, cudaStream_t stream) {
  if (!in || !w || !bias || !out || B < 0 || C <= 0 || O <= 0 || kh <= 0 || kw <= 0 || H % kh ||
      W % kw)
    return VT_ERR_ARG;
  const long long total = static_cast<long long>(B) * O * (H / kh) * (W / kw);
  if (total == 0) return VT_OK;
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  if (dtype == VT_F32)
    conv2d_nchw_kernel<float><<<grid, 256, 0, stream>>>(
        static_cast<const float*>(in), static_cast<const float*>(w),
        static_cast<const float*>(bias), static_cast<float*>(out), B, C, H, W, O, kh, kw);
  else if (dtype == VT_BF16)
    conv2d_nchw_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(
        static_cast<const __nv_bfloat16*>(in), static_cast<const __nv_bfloat16*>(w),
        static_cast<const __nv_bfloat16*>(bias), static_cast<__nv_bfloat16*>(out), B, C, H, W, O,
        kh, kw);
  else
    return VT_ERR_DTYPE;
  return static_cast<int>(cudaGetLastError());
}

}  // namespace vt
