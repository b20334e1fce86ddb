// K2a: patch gather — pixels -> padded bf16 patch rows, the A operand of the patch-embedding GEMM (K2b = the
// 2-CTA tcgen05 GEMM of gemm2_sm100.cu in token mode).  Bandwidth-bound, every pixel is read ONCE:
//
//   A[b, 0, :]        = 0                                   (CLS slot: the GEMM adds bias + (cls + pos[0] - bias))
//   A[b, 1 + p, k]    = pixel k of patch p of image b       k = (c, i, j) for NCHW fp32 / bf16 pixels,
//                                                           k = (i, j, c) for NHWC uint8 pixels
//   A[b, t, :]        = 0 for n < t < Tpad,  A[.., k] = 0 for K <= k < Kpad
//
// Tpad = tokens rounded up to 32: no 32-row tile of the GEMM's epilogue straddles two images, so its output and
// position-table coordinates are (token, image) and TMA clips the padding rows.  Round 1's single kernel
// (patch_embed_sm100.cu, kept for head widths that are not a multiple of 8 and as the A/B baseline) gathered the
// pixels once per 256-column block of the output — three times for ViT-B — and ran at 172 us (tensor pipe 17 %,
// DRAM 8 %); gather + GEMM need one pass over the pixels and one tensor-bound GEMM.
// Replaces the patch extraction inside conv2d_kernel (vit/kernels/conv2d.py:19-97) / patching_kernel
// (vit/kernels/patching.py:54-92).
#include "common.cuh"

namespace vt {

namespace {

struct GatherParams {
  const void* pixels;
  __nv_bfloat16* out;
  int B, C, H, W, P, grid_w, n_patches, K, Kpad, Tpad;
  long long total_chunks;    // B * Tpad * Kpad / 8
};

__device__ __forceinline__ float gpx(float v) { return v; }
__device__ __forceinline__ float gpx(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float gpx(uint8_t v) { return static_cast<float>(v); }

// one thread = one 16-byte chunk (8 bf16) of A; blockIdx.x = token row, blockIdx.y = image: no division by the row
// length or the token count (the first version decoded a flat 64-bit chunk index with four 64-bit divisions per
// chunk and ran at 44 us for the C2 batch, issue-bound: 77 % issue slots, DRAM 35 %; now ~40.  Staging whole image
// rows through shared memory so that both sides are fully coalesced gains another 1.6 us only: not kept)
template <typename TPix, bool kVec>
__global__ void __launch_bounds__(128)
patch_gather_kernel(const GatherParams p) {
  constexpr bool kNHWC = sizeof(TPix) == 1;
  const int chunks_per_row = p.Kpad >> 3;
  const int t = blockIdx.x;
  const int b = blockIdx.y;
  const int patch = t - 1;
  const int py = patch / p.grid_w, px = patch - py * p.grid_w;      // block-uniform
  const bool real_row = t >= 1 && t <= p.n_patches;
  const TPix* img = static_cast<const TPix*>(p.pixels) + static_cast<long long>(b) * p.C * p.H * p.W;
  uint4* out_row = reinterpret_cast<uint4*>(p.out) + (static_cast<long long>(b) * p.Tpad + t) * chunks_per_row;
  for (int kc = threadIdx.x; kc < chunks_per_row; kc += blockDim.x) {
    const int k0 = kc << 3;
    uint4 o = make_uint4(0u, 0u, 0u, 0u);
    if (real_row && k0 < p.K) {
      if constexpr (kVec && kNHWC) {
        const int PC = p.P * p.C;                 // bytes of one patch row; PC % 8 == 0
        const int i = k0 / PC, rem = k0 - i * PC;
        const uint2 v = __ldg(reinterpret_cast<const uint2*>(
            img + (static_cast<long long>(py * p.P + i) * p.W + px * p.P) * p.C + rem));
        auto f = [](uint32_t w, int s) { return static_cast<float>((w >> (8 * s)) & 0xFFu); };
        o = make_uint4(pack_bf16x2(f(v.x, 0), f(v.x, 1)), pack_bf16x2(f(v.x, 2), f(v.x, 3)),
                       pack_bf16x2(f(v.y, 0), f(v.y, 1)), pack_bf16x2(f(v.y, 2), f(v.y, 3)));
      } else if constexpr (kVec) {
        const int PP = p.P * p.P;
        const int c = k0 / PP, rem = k0 - c * PP;
        const int i = rem / p.P, j = rem - i * p.P;   // P % 8 == 0: the 8 pixels stay inside one patch row
        const TPix* src = img + (static_cast<long long>(c) * p.H + py * p.P + i) * p.W + px * p.P + j;
        if constexpr (sizeof(TPix) == 2) {
          o = __ldg(reinterpret_cast<const uint4*>(src));
        } else {
          const float4 a = __ldg(reinterpret_cast<const float4*>(src));
          const float4 c4 = __ldg(reinterpret_cast<const float4*>(src) + 1);
          o = make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(c4.x, c4.y), pack_bf16x2(c4.z, c4.w));
        }
      } else {
        float e[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int k = k0 + u;
          e[u] = 0.f;
          if (k < p.K) {
            if constexpr (kNHWC) {
              const int PC = p.P * p.C;
              const int i = k / PC, rem = k - i * PC;
              e[u] = gpx(img[(static_cast<long long>(py * p.P + i) * p.W + px * p.P) * p.C + rem]);
            } else {
              const int PP = p.P * p.P;
              const int c = k / PP, rem = k - c * PP;
              const int i = rem / p.P, j = rem - i * p.P;
              e[u] = gpx(img[(static_cast<long long>(c) * p.H + py * p.P + i) * p.W + px * p.P + j]);
            }
          }
        }
        o = make_uint4(pack_bf16x2(e[0], e[1]), pack_bf16x2(e[2], e[3]), pack_bf16x2(e[4], e[5]), pack_bf16x2(e[6], e[7]));
      }
    }
    out_row[kc] = o;
  }
}

template <typename TPix, bool kVec>
int launch_gather(const GatherParams& p, cudaStream_t stream) {
  if (p.B > 65535) return VT_ERR_UNSUPPORTED;
  patch_gather_kernel<TPix, kVec><<<dim3(p.Tpad, p.B), 128, 0, stream>>>(p);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace

// pixels: [B, C, H, W] (f32 | bf16) or [B, H, W, C] (VT_U8); the patch grid is (H / P) x (W / P) rounded down, the
// pixels of the last H % P rows and W % P columns belong to no patch (a stride-P convolution drops them too).
// out: bf16 [B, Tpad, Kpad] (Kpad % 8 == 0, Tpad >= n_patches + 1), 16-byte aligned.
int patch_gather(const void* pixels, int pix_dtype, void* out, int B, int C, int H, int W, int P, int Tpad, int Kpad,
                 cudaStream_t stream) {
  if (!pixels || !out || B <= 0 || C <= 0 || P <= 0 || H < P || W < P) return VT_ERR_ARG;
  GatherParams p;
  p.pixels = pixels;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.B = B; p.C = C; p.H = H; p.W = W; p.P = P;
  p.grid_w = W / P;
  p.n_patches = (H / P) * p.grid_w;
  p.K = C * P * P;
  p.Kpad = Kpad;
  p.Tpad = Tpad;
  if ((Kpad % 8) || Kpad < p.K || Tpad < p.n_patches + 1) return VT_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(pixels) | reinterpret_cast<uintptr_t>(out)) & 15) return VT_ERR_ALIGN;
  p.total_chunks = static_cast<long long>(B) * Tpad * (Kpad / 8);
  // vector loads need every 8-element chunk inside one patch row and 8-element aligned: image rows of a multiple of
  // 8 elements (W * C bytes for NHWC, W for NCHW) then keep every row, plane and image start aligned too
  if (pix_dtype == VT_U8) {
    const bool vec = ((P * C) % 8 == 0) && ((W * C) % 8 == 0);
    return vec ? launch_gather<uint8_t, true>(p, stream) : launch_gather<uint8_t, false>(p, stream);
  }
  const bool vec = (P % 8 == 0) && (W % 8 == 0);
  if (pix_dtype == VT_BF16)
    return vec ? launch_gather<__nv_bfloat16, true>(p, stream) : launch_gather<__nv_bfloat16, false>(p, stream);
  if (pix_dtype == VT_F32) return vec ? launch_gather<float, true>(p, stream) : launch_gather<float, false>(p, stream);
  return VT_ERR_DTYPE;
}

}  // namespace vt
