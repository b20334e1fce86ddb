// Masked image modeling head (vt_mim_reconstruct): PixelShuffle of the decoder's 1x1-convolution output back into an
// image, and HF ViTForMaskedImageModeling's masked L1 loss against the input pixels in the same pass.
//
//   rec[b, c, y*s + i, x*s + j] = dec[b, 1 + y*gw + x, (c*s + i)*s + j]
//   loss = sum_{masked patches} |pixel - rec| / (masked patches * s^2 + 1e-5) / C
//
// One block per (image, patch): it reads the patch's decoder row once (coalesced), writes s contiguous elements per
// (channel, pixel row) of the image, and, for a masked patch, reduces |pixel - rec| over its s^2 C pixels in a fixed
// order (strided per-thread sums, xor-shuffle warp sums, warps summed in index order) into partial[patch].  A second
// single-block launch sums the partials in fixed order in fp64, so the loss is bit-identical from call to call and
// under graph replay, with no atomics and no host synchronisation.
#include "common.cuh"

namespace vt {

namespace {

constexpr int kThreads = 256;
constexpr int kFinalThreads = 1024;

__device__ __forceinline__ float ldv(const float* p) { return *p; }
__device__ __forceinline__ float ldv(const __nv_bfloat16* p) { return __bfloat162float(*p); }

struct MimParams {
  const void* dec;
  void* rec;
  const void* pixels;
  const float* norm;
  const uint8_t* mask;
  float* partial;
  float rescale;
  int C, gh, gw, s;
};

template <typename T, typename TPix, bool kLoss>
__global__ void __launch_bounds__(kThreads)
mim_reconstruct_kernel(const MimParams p) {
  const long long n = static_cast<long long>(p.gh) * p.gw;
  const long long blk = blockIdx.x;
  const long long b = blk / n;
  const int patch = static_cast<int>(blk - b * n);
  const int y = patch / p.gw, x = patch - y * p.gw;
  const int ss = p.s * p.s;
  const int L = ss * p.C;
  const long long Hr = static_cast<long long>(p.gh) * p.s, Wr = static_cast<long long>(p.gw) * p.s;
  const T* src = static_cast<const T*>(p.dec) + (b * (n + 1) + 1 + patch) * L;
  T* rec = static_cast<T*>(p.rec);
  const bool masked = kLoss && p.mask[blk] != 0;                // block-uniform
  float acc = 0.f;
  for (int e = threadIdx.x; e < L; e += kThreads) {
    const int c = e / ss, r = e - c * ss;
    const int i = r / p.s, j = r - i * p.s;
    const long long yy = static_cast<long long>(y) * p.s + i, xx = static_cast<long long>(x) * p.s + j;
    const T v = src[e];
    rec[((b * p.C + c) * Hr + yy) * Wr + xx] = v;
    if (masked) {
      float px;
      if constexpr (sizeof(TPix) == 1) {
        const uint8_t u = static_cast<const uint8_t*>(p.pixels)[((b * Hr + yy) * Wr + xx) * p.C + c];
        px = (static_cast<float>(u) * p.rescale - p.norm[c]) / p.norm[p.C + c];
      } else {
        px = ldv(static_cast<const TPix*>(p.pixels) + ((b * p.C + c) * Hr + yy) * Wr + xx);
      }
      acc += fabsf(px - ldv(&v));
    }
  }
  if constexpr (kLoss) {
    __shared__ float warp_acc[kThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) warp_acc[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < kThreads / 32; ++w) t += warp_acc[w];
      p.partial[blk] = masked ? t : 0.f;
    }
  }
}

__global__ void __launch_bounds__(kFinalThreads)
mim_loss_kernel(const float* __restrict__ partial, const uint8_t* __restrict__ mask, long long count, int ss, int C,
                float* __restrict__ loss) {
  __shared__ double sums[kFinalThreads];
  __shared__ long long hits[kFinalThreads];
  double acc = 0.0;
  long long cnt = 0;
  for (long long i = threadIdx.x; i < count; i += kFinalThreads) {
    acc += static_cast<double>(partial[i]);
    cnt += mask[i] != 0;
  }
  sums[threadIdx.x] = acc;
  hits[threadIdx.x] = cnt;
  __syncthreads();
  for (int half = kFinalThreads / 2; half > 0; half >>= 1) {
    if (threadIdx.x < half) {
      sums[threadIdx.x] += sums[threadIdx.x + half];
      hits[threadIdx.x] += hits[threadIdx.x + half];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double pixels = static_cast<double>(hits[0]) * ss;
    *loss = static_cast<float>(sums[0] / (pixels + 1e-5) / C);
  }
}

template <typename T, typename TPix, bool kLoss>
int launch_mim(const MimParams& p, long long blocks, cudaStream_t stream) {
  mim_reconstruct_kernel<T, TPix, kLoss><<<static_cast<unsigned>(blocks), kThreads, 0, stream>>>(p);
  return static_cast<int>(cudaGetLastError());
}

template <typename T>
int launch_mim_pix(const MimParams& p, int pix_dtype, bool with_loss, long long blocks, cudaStream_t stream) {
  if (!with_loss) return launch_mim<T, float, false>(p, blocks, stream);
  if (pix_dtype == VT_F32) return launch_mim<T, float, true>(p, blocks, stream);
  if (pix_dtype == VT_BF16) return launch_mim<T, __nv_bfloat16, true>(p, blocks, stream);
  if (pix_dtype == VT_U8) return launch_mim<T, uint8_t, true>(p, blocks, stream);
  return VT_ERR_DTYPE;
}

}  // namespace

int mim_reconstruct(const void* dec, void* rec, int dtype, int B, int C, int gh, int gw, int s, const void* pixels,
                    int pix_dtype, const float* norm, float rescale, const void* mask, float* partial, float* loss,
                    cudaStream_t stream) {
  if (!dec || !rec || B <= 0 || C <= 0 || gh <= 0 || gw <= 0 || s <= 0) return VT_ERR_ARG;
  const bool with_loss = loss != nullptr;
  if (with_loss && (!pixels || !mask || !partial || (pix_dtype == VT_U8 && !norm))) return VT_ERR_ARG;
  const long long blocks = static_cast<long long>(B) * gh * gw;
  if (blocks > 0x7fffffffLL || static_cast<long long>(s) * s * C > 0x7fffffffLL) return VT_ERR_UNSUPPORTED;
  MimParams p;
  p.dec = dec;
  p.rec = rec;
  p.pixels = pixels;
  p.norm = norm;
  p.mask = static_cast<const uint8_t*>(mask);
  p.partial = partial;
  p.rescale = rescale;
  p.C = C; p.gh = gh; p.gw = gw; p.s = s;
  int rc;
  if (dtype == VT_F32) rc = launch_mim_pix<float>(p, pix_dtype, with_loss, blocks, stream);
  else if (dtype == VT_BF16) rc = launch_mim_pix<__nv_bfloat16>(p, pix_dtype, with_loss, blocks, stream);
  else return VT_ERR_DTYPE;
  if (rc || !with_loss) return rc;
  mim_loss_kernel<<<1, kFinalThreads, 0, stream>>>(partial, p.mask, blocks, s * s, C, loss);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace vt
