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
#include "../../include/vitb200_ragged.h"

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

// One 16-byte chunk of a patch row: elements k0 .. k0 + 7 (k0 < K, k0 % 8 == 0) of patch (py, px) of one image, the
// elements >= K zero.  The addressing of both gathers (the batched one below and the ragged one of
// vt_patch_embed_ragged_gather).  kVec: 8-element loads, which need P % 8 == 0 and W % 8 == 0 (NCHW) / P * C and
// W * C multiples of 8 (NHWC), and a 16-byte aligned image.
template <typename TPix, bool kVec>
__device__ __forceinline__ uint4 gather_chunk(const TPix* img, int C, int H, int W, int P, int K, int py, int px,
                                              int k0) {
  constexpr bool kNHWC = sizeof(TPix) == 1;
  if constexpr (kVec && kNHWC) {
    const int PC = P * C;                     // bytes of one patch row; PC % 8 == 0
    const int i = k0 / PC, rem = k0 - i * PC;
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(img + (static_cast<long long>(py * P + i) * W + px * P) * C + rem));
    auto f = [](uint32_t w, int s) { return static_cast<float>((w >> (8 * s)) & 0xFFu); };
    return make_uint4(pack_bf16x2(f(v.x, 0), f(v.x, 1)), pack_bf16x2(f(v.x, 2), f(v.x, 3)),
                      pack_bf16x2(f(v.y, 0), f(v.y, 1)), pack_bf16x2(f(v.y, 2), f(v.y, 3)));
  } else if constexpr (kVec) {
    const int PP = P * P;
    const int c = k0 / PP, rem = k0 - c * PP;
    const int i = rem / P, j = rem - i * P;   // P % 8 == 0: the 8 pixels stay inside one patch row
    const TPix* src = img + (static_cast<long long>(c) * H + py * P + i) * W + px * P + j;
    if constexpr (sizeof(TPix) == 2) {
      return __ldg(reinterpret_cast<const uint4*>(src));
    } else {
      const float4 a = __ldg(reinterpret_cast<const float4*>(src));
      const float4 c4 = __ldg(reinterpret_cast<const float4*>(src) + 1);
      return make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(c4.x, c4.y), pack_bf16x2(c4.z, c4.w));
    }
  } else {
    float e[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int k = k0 + u;
      e[u] = 0.f;
      if (k < K) {
        if constexpr (kNHWC) {
          const int PC = P * C;
          const int i = k / PC, rem = k - i * PC;
          e[u] = gpx(img[(static_cast<long long>(py * P + i) * W + px * P) * C + rem]);
        } else {
          const int PP = P * P;
          const int c = k / PP, rem = k - c * PP;
          const int i = rem / P, j = rem - i * P;
          e[u] = gpx(img[(static_cast<long long>(c) * H + py * P + i) * W + px * P + j]);
        }
      }
    }
    return make_uint4(pack_bf16x2(e[0], e[1]), pack_bf16x2(e[2], e[3]), pack_bf16x2(e[4], e[5]), pack_bf16x2(e[6], e[7]));
  }
}

// one thread = one 16-byte chunk (8 bf16) of A; blockIdx.x = token row, blockIdx.y = image: no division by the row
// length or the token count (the first version decoded a flat 64-bit chunk index with four 64-bit divisions per
// chunk and ran at 44 us for the C2 batch, issue-bound: 77 % issue slots, DRAM 35 %; now ~40.  Staging whole image
// rows through shared memory so that both sides are fully coalesced gains another 1.6 us only: not kept)
template <typename TPix, bool kVec>
__global__ void __launch_bounds__(128)
patch_gather_kernel(const GatherParams p) {
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
    if (real_row && k0 < p.K) o = gather_chunk<TPix, kVec>(img, p.C, p.H, p.W, p.P, p.K, py, px, k0);
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

// ------------------------------------------------------------------------------------------------ ragged batch
// Images of different sizes in one launch (vt_patch_embed_ragged_gather): one block per packed output row.  The row's
// image is found by a binary search over the descriptors' first rows (log2(images) cached loads, block-uniform); the
// block writes the row's patch pixels (gather_chunk, the batched kernel's addressing) and the image's position row, the
// residual of the embedding GEMM.  No row padding: the GEMM runs in plain mode over the packed rows, whose epilogue
// adds bias + residual in the same order as token mode, so every image comes out as it does from its own call.
namespace {

struct RaggedParams {
  const vt_ragged_image* images;
  __nv_bfloat16* patches;
  __nv_bfloat16* table;
  int n_images, C, P, K, Kpad, D;
};

template <typename TPix>
__global__ void __launch_bounds__(128)
patch_gather_ragged_kernel(const RaggedParams p) {
  constexpr bool kNHWC = sizeof(TPix) == 1;
  const long long row = blockIdx.x;
  int lo = 0, hi = p.n_images - 1;                  // last image with row0 <= row
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(&p.images[mid].row0) <= row) lo = mid; else hi = mid - 1;
  }
  const vt_ragged_image* d = p.images + lo;
  const long long row0 = __ldg(&d->row0);
  const int H = __ldg(&d->height), W = __ldg(&d->width);
  const long long t64 = row - row0;
  const bool covered = t64 >= 0 && t64 < __ldg(&d->tokens);
  const int t = covered ? static_cast<int>(t64) : 0;
  const int grid_w = W / p.P;
  const int n_patches = (H / p.P) * grid_w;
  const bool real_row = covered && t >= 1 && t <= n_patches;
  const int patch = real_row ? t - 1 : 0;
  const int py = patch / grid_w, px = patch - py * grid_w;
  const TPix* img = static_cast<const TPix*>(d->pixels);
  const bool aligned = (reinterpret_cast<uintptr_t>(img) & 15) == 0;
  const bool vec = aligned && (kNHWC ? ((p.P * p.C) % 8 == 0 && (W * p.C) % 8 == 0) : (p.P % 8 == 0 && W % 8 == 0));

  const int chunks_per_row = p.Kpad >> 3;
  uint4* out_row = reinterpret_cast<uint4*>(p.patches) + row * chunks_per_row;
  for (int kc = threadIdx.x; kc < chunks_per_row; kc += blockDim.x) {
    const int k0 = kc << 3;
    uint4 o = make_uint4(0u, 0u, 0u, 0u);
    if (real_row && k0 < p.K)
      o = vec ? gather_chunk<TPix, true>(img, p.C, H, W, p.P, p.K, py, px, k0)
              : gather_chunk<TPix, false>(img, p.C, H, W, p.P, p.K, py, px, k0);
    out_row[kc] = o;
  }

  const int dchunks = p.D >> 3;
  const __nv_bfloat16* pos = static_cast<const __nv_bfloat16*>(d->pos) + static_cast<long long>(t) * p.D;
  uint4* tab_row = reinterpret_cast<uint4*>(p.table) + row * dchunks;
  const bool pos_aligned = (reinterpret_cast<uintptr_t>(d->pos) & 15) == 0;
  for (int c = threadIdx.x; c < dchunks; c += blockDim.x) {
    uint4 o = make_uint4(0u, 0u, 0u, 0u);
    if (covered) {
      if (pos_aligned) {
        o = __ldg(reinterpret_cast<const uint4*>(pos) + c);
      } else {
        const unsigned short* s = reinterpret_cast<const unsigned short*>(pos) + (c << 3);
        uint32_t w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) w[u] = static_cast<uint32_t>(__ldg(s + 2 * u)) | (static_cast<uint32_t>(__ldg(s + 2 * u + 1)) << 16);
        o = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
    tab_row[c] = o;
  }
}

}  // namespace

int patch_gather_ragged(const void* images, int n_images, int pix_dtype, int C, int P, void* patches, long long ldw,
                        void* table, int D, long long M, cudaStream_t stream) {
  if (!images || !patches || !table || n_images <= 0 || C <= 0 || P <= 0 || D <= 0 || M <= 0) return VT_ERR_ARG;
  if (M > 0x7fffffffLL) return VT_ERR_UNSUPPORTED;
  const long long K = static_cast<long long>(C) * P * P;
  if (ldw < K || ldw > 0x7fffffffLL) return VT_ERR_ARG;
  if ((ldw % 8) || (D % 8)) return VT_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(patches) | reinterpret_cast<uintptr_t>(table)) & 15) return VT_ERR_ALIGN;
  RaggedParams p;
  p.images = static_cast<const vt_ragged_image*>(images);
  p.patches = static_cast<__nv_bfloat16*>(patches);
  p.table = static_cast<__nv_bfloat16*>(table);
  p.n_images = n_images; p.C = C; p.P = P; p.K = static_cast<int>(K); p.Kpad = static_cast<int>(ldw); p.D = D;
  const dim3 grid(static_cast<unsigned int>(M));
  if (pix_dtype == VT_U8) patch_gather_ragged_kernel<uint8_t><<<grid, 128, 0, stream>>>(p);
  else if (pix_dtype == VT_BF16) patch_gather_ragged_kernel<__nv_bfloat16><<<grid, 128, 0, stream>>>(p);
  else if (pix_dtype == VT_F32) patch_gather_ragged_kernel<float><<<grid, 128, 0, stream>>>(p);
  else return VT_ERR_DTYPE;
  return static_cast<int>(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------ masked batch
// bool_masked_pos (vt_patch_embed_masked_gather): one block per unpadded output row (blockIdx.x = token, blockIdx.y =
// image).  A masked patch's row is zero and its table row carries mask_token + pos - bias, so the plain-mode GEMM's
// bias + residual epilogue turns it into mask_token + pos; an unmasked row is the batched gather's row and pos[t].
namespace {

struct MaskedParams {
  const void* pixels;
  const uint8_t* mask;
  const uint4* pos;
  const uint4* posm;
  uint4* patches;
  uint4* table;
  int C, H, W, P, grid_w, n_patches, K, Kpad, D;
};

template <typename TPix, bool kVec>
__global__ void __launch_bounds__(128)
patch_gather_masked_kernel(const MaskedParams p) {
  const int t = blockIdx.x;
  const int b = blockIdx.y;
  const int N = p.n_patches + 1;
  const int patch = t > 0 ? t - 1 : 0;
  const bool masked = t > 0 && p.mask[static_cast<long long>(b) * p.n_patches + patch] != 0;   // block-uniform
  const bool real_row = t > 0 && !masked;
  const int py = patch / p.grid_w, px = patch - py * p.grid_w;
  const TPix* img = static_cast<const TPix*>(p.pixels) + static_cast<long long>(b) * p.C * p.H * p.W;
  const long long row = static_cast<long long>(b) * N + t;

  const int chunks_per_row = p.Kpad >> 3;
  uint4* out_row = p.patches + row * chunks_per_row;
  for (int kc = threadIdx.x; kc < chunks_per_row; kc += blockDim.x) {
    const int k0 = kc << 3;
    uint4 o = make_uint4(0u, 0u, 0u, 0u);
    if (real_row && k0 < p.K) o = gather_chunk<TPix, kVec>(img, p.C, p.H, p.W, p.P, p.K, py, px, k0);
    out_row[kc] = o;
  }

  const int dchunks = p.D >> 3;
  const uint4* src = (masked ? p.posm : p.pos) + static_cast<long long>(t) * dchunks;
  uint4* tab_row = p.table + row * dchunks;
  for (int c = threadIdx.x; c < dchunks; c += blockDim.x) tab_row[c] = __ldg(src + c);
}

template <typename TPix, bool kVec>
int launch_masked(const MaskedParams& p, int B, cudaStream_t stream) {
  patch_gather_masked_kernel<TPix, kVec><<<dim3(p.n_patches + 1, B), 128, 0, stream>>>(p);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace

int patch_gather_masked(const void* pixels, int pix_dtype, const void* mask, const void* pos, const void* posm,
                        void* patches, long long ldw, void* table, int B, int C, int H, int W, int P, int D,
                        cudaStream_t stream) {
  if (!pixels || !mask || !pos || !posm || !patches || !table || B <= 0 || C <= 0 || P <= 0 || D <= 0 || H < P ||
      W < P)
    return VT_ERR_ARG;
  const long long K = static_cast<long long>(C) * P * P;
  if (ldw < K || ldw > 0x7fffffffLL) return VT_ERR_ARG;
  if ((ldw % 8) || (D % 8)) return VT_ERR_ALIGN;
  const long long n = static_cast<long long>(H / P) * (W / P);
  if (B > 65535 || static_cast<long long>(B) * (n + 1) > 0x7fffffffLL) return VT_ERR_UNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(pixels) | reinterpret_cast<uintptr_t>(patches) | reinterpret_cast<uintptr_t>(table) |
       reinterpret_cast<uintptr_t>(pos) | reinterpret_cast<uintptr_t>(posm)) & 15)
    return VT_ERR_ALIGN;
  MaskedParams p;
  p.pixels = pixels;
  p.mask = static_cast<const uint8_t*>(mask);
  p.pos = static_cast<const uint4*>(pos);
  p.posm = static_cast<const uint4*>(posm);
  p.patches = static_cast<uint4*>(patches);
  p.table = static_cast<uint4*>(table);
  p.C = C; p.H = H; p.W = W; p.P = P;
  p.grid_w = W / P;
  p.n_patches = static_cast<int>(n);
  p.K = static_cast<int>(K);
  p.Kpad = static_cast<int>(ldw);
  p.D = D;
  // the vector-load conditions of patch_gather
  if (pix_dtype == VT_U8) {
    const bool vec = ((P * C) % 8 == 0) && ((W * C) % 8 == 0);
    return vec ? launch_masked<uint8_t, true>(p, B, stream) : launch_masked<uint8_t, false>(p, B, stream);
  }
  const bool vec = (P % 8 == 0) && (W % 8 == 0);
  if (pix_dtype == VT_BF16)
    return vec ? launch_masked<__nv_bfloat16, true>(p, B, stream) : launch_masked<__nv_bfloat16, false>(p, B, stream);
  if (pix_dtype == VT_F32) return vec ? launch_masked<float, true>(p, B, stream) : launch_masked<float, false>(p, B, stream);
  return VT_ERR_DTYPE;
}

}  // namespace vt
