// vt_resize_u8 / vt_resize_u8_list: PIL's Image.resize (BILINEAR, BICUBIC) of uint8 HWC images on the device, byte
// for byte, with the coefficient tables of include/vitb200_preprocess.h built on the host.
//
// A CTA owns one (image, band of kTY output rows, tile of kTX output columns).  The band's input rows are
// [start of its first row, start + count of its last row) of the height table.  It walks them in chunks of kChunk:
//   1. the width pass of the chunk's rows for the tile's columns, rounded to uint8 (PIL's intermediate) in shared
//      memory; a thread keeps one column and steps over the rows;
//   2. every output pixel of the tile adds the chunk's share of its height taps to its int32 sum (thread = pixel).
// Images that PIL resizes height first (more than 100 times taller than wide, height shrinking) take the same
// schedule with the axes exchanged: chunks of the tile's input columns, the height pass into shared memory, then the
// width taps.
// The sums are exact integers, so chunking gives PIL's bytes, and shared memory stays kChunk * kTX * C bytes however
// large the downscale.  At the end each thread shifts, clamps and stores its pixel's C bytes.
// Memory accesses: source sample indices are start + j with j < count of a table entry only (rows through the band's
// range above); pixel addresses are 64-bit; a thread writes only its own (image, oy < out_h, ox < out_w, c < C).
// Plain byte loads: images of odd widths start anywhere.
#include "../../include/vitb200_preprocess.h"
#include "common.cuh"

namespace vt {

namespace {

constexpr int kTX = 32;                   // output columns per CTA (one warp-wide row)
constexpr int kTY = 8;                    // output rows per CTA
constexpr int kThreads = kTX * kTY;       // one output pixel per thread
constexpr int kChunk = 32;                // input rows per shared-memory chunk
constexpr int kMaxGridY = 65535;          // images per launch
static_assert(kChunk == kTX, "a thread's first-pass column / row is its output pixel's");

struct ResizeParams {
  const uint8_t* src;                     // batch form
  long long batch_stride;
  const int32_t* htab;
  const int32_t* vtab;
  int H, W, hk, vk;
  const vt_resize_image* images;          // list form
  const int32_t* tables;
  uint8_t* out;
  int out_h, out_w, col_tiles, image0;
};

__device__ __forceinline__ uint8_t clip8(int v) {
  v >>= 22;
  return static_cast<uint8_t>(v < 0 ? 0 : (v > 255 ? 255 : v));
}

template <int C, bool kList>
__global__ void __launch_bounds__(kThreads, 6)
vt_resize_u8_kernel(const ResizeParams p) {
  __shared__ uint8_t inter[kChunk * kTX * C];
  const long long img = static_cast<long long>(p.image0) + blockIdx.y;
  const int band = blockIdx.x / p.col_tiles;
  const int tile = blockIdx.x - band * p.col_tiles;
  const uint8_t* src;
  const int32_t* htab;
  const int32_t* vtab;
  int H, W, hk, vk;
  if constexpr (kList) {
    const vt_resize_image* d = p.images + img;
    src = static_cast<const uint8_t*>(d->pixels);
    H = d->height;
    W = d->width;
    hk = d->hk;
    vk = d->vk;
    htab = p.tables + d->htab;
    vtab = p.tables + d->vtab;
  } else {
    src = p.src + img * p.batch_stride;
    H = p.H;
    W = p.W;
    hk = p.hk;
    vk = p.vk;
    htab = p.htab;
    vtab = p.vtab;
  }
  const long long hs = 2 + hk, vs = 2 + vk;          // table row lengths in int32
  const long long row_bytes = static_cast<long long>(W) * C;
  const int oy0 = band * kTY, ox0 = tile * kTX;
  // this thread's output pixel and its two table entries; it is also the width-pass column (height-first: the
  // height-pass row) of the first pass, since kTX == kChunk and the thread's column / row do not change
  const int ty = threadIdx.x / kTX, tx = threadIdx.x % kTX;
  const int oy = oy0 + ty, ox = ox0 + tx;
  const bool row_ok = oy < p.out_h, col_ok = ox < p.out_w;
  const int32_t* he = htab + (col_ok ? ox : 0) * hs;
  const int32_t* ve = vtab + (row_ok ? oy : 0) * vs;
  const int h_start = col_ok ? __ldg(he) : 0, h_count = col_ok ? __ldg(he + 1) : 0;
  const int v_start = row_ok ? __ldg(ve) : 0, v_count = row_ok ? __ldg(ve + 1) : 0;
  int acc[C];
#pragma unroll
  for (int c = 0; c < C; ++c) acc[c] = 1 << 21;

  // PIL >= 12 resizes an image more than 100 times taller than wide height first when the height shrinks
  // (Image.resize); every other image width first.  Block-uniform.
  if (!(H > 100LL * W && p.out_h < H)) {
    const int oy_last = min(oy0 + kTY, p.out_h) - 1;
    const int ylo = __ldg(vtab + oy0 * vs);
    const int yhi = __ldg(vtab + oy_last * vs) + __ldg(vtab + oy_last * vs + 1);
    for (int y0 = ylo; y0 < yhi; y0 += kChunk) {
      const int rows = min(kChunk, yhi - y0);
      // width pass of input rows y0 .. y0 + rows for column ox -> inter[r][tx]
      if (col_ok) {
        for (int r = ty; r < rows; r += kTY) {
          const uint8_t* px = src + static_cast<long long>(y0 + r) * row_bytes + static_cast<long long>(h_start) * C;
          int h[C];
#pragma unroll
          for (int c = 0; c < C; ++c) h[c] = 1 << 21;
#pragma unroll 1
          for (int j = 0; j < h_count; ++j) {
            const int w = __ldg(he + 2 + j);
#pragma unroll
            for (int c = 0; c < C; ++c) h[c] += static_cast<int>(__ldg(px + j * C + c)) * w;
          }
#pragma unroll
          for (int c = 0; c < C; ++c) inter[(r * kTX + tx) * C + c] = clip8(h[c]);
        }
      }
      __syncthreads();
      // height taps of pixel (oy, ox) inside the chunk
      if (row_ok && col_ok) {
        const int lo = max(v_start, y0), hi = min(v_start + v_count, y0 + rows);
        for (int y = lo; y < hi; ++y) {
          const int w = __ldg(ve + 2 + (y - v_start));
          const uint8_t* s = inter + ((y - y0) * kTX + tx) * C;
#pragma unroll
          for (int c = 0; c < C; ++c) acc[c] += static_cast<int>(s[c]) * w;
        }
      }
      __syncthreads();
    }
  } else {
    const int ox_last = min(ox0 + kTX, p.out_w) - 1;
    const int xlo = __ldg(htab + ox0 * hs);
    const int xhi = __ldg(htab + ox_last * hs) + __ldg(htab + ox_last * hs + 1);
    for (int x0 = xlo; x0 < xhi; x0 += kChunk) {
      const int cols = min(kChunk, xhi - x0);
      // height pass of input columns x0 .. x0 + cols for row oy -> inter[ty][i]
      if (row_ok && tx < cols) {
        const uint8_t* px = src + static_cast<long long>(v_start) * row_bytes + static_cast<long long>(x0 + tx) * C;
        int h[C];
#pragma unroll
        for (int c = 0; c < C; ++c) h[c] = 1 << 21;
#pragma unroll 1
        for (int j = 0; j < v_count; ++j) {
          const int w = __ldg(ve + 2 + j);
#pragma unroll
          for (int c = 0; c < C; ++c) h[c] += static_cast<int>(__ldg(px + j * row_bytes + c)) * w;
        }
#pragma unroll
        for (int c = 0; c < C; ++c) inter[(ty * kChunk + tx) * C + c] = clip8(h[c]);
      }
      __syncthreads();
      // width taps of pixel (oy, ox) inside the chunk
      if (row_ok && col_ok) {
        const int lo = max(h_start, x0), hi = min(h_start + h_count, x0 + cols);
        for (int x = lo; x < hi; ++x) {
          const int w = __ldg(he + 2 + (x - h_start));
          const uint8_t* s = inter + (ty * kChunk + (x - x0)) * C;
#pragma unroll
          for (int c = 0; c < C; ++c) acc[c] += static_cast<int>(s[c]) * w;
        }
      }
      __syncthreads();
    }
  }
  if (row_ok && col_ok) {
    uint8_t* o = p.out + ((img * p.out_h + oy) * p.out_w + ox) * C;
#pragma unroll
    for (int c = 0; c < C; ++c) o[c] = clip8(acc[c]);
  }
}

template <int C, bool kList>
int launch_resize(ResizeParams p, int n_images, cudaStream_t stream) {
  const int bands = (p.out_h + kTY - 1) / kTY;
  p.col_tiles = (p.out_w + kTX - 1) / kTX;
  for (int i0 = 0; i0 < n_images; i0 += kMaxGridY) {
    p.image0 = i0;
    const int n = min(kMaxGridY, n_images - i0);
    vt_resize_u8_kernel<C, kList><<<dim3(static_cast<unsigned>(bands) * p.col_tiles, n), kThreads, 0, stream>>>(p);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return static_cast<int>(e);
  }
  return 0;
}

template <bool kList>
int launch_resize_c(const ResizeParams& p, int C, int n_images, cudaStream_t stream) {
  switch (C) {
    case 1: return launch_resize<1, kList>(p, n_images, stream);
    case 2: return launch_resize<2, kList>(p, n_images, stream);
    case 3: return launch_resize<3, kList>(p, n_images, stream);
    default: return launch_resize<4, kList>(p, n_images, stream);
  }
}

// CTAs per image fit the grid's x dimension
bool grid_fits(int out_h, int out_w) {
  const long long ctas = static_cast<long long>((out_h + kTY - 1) / kTY) * ((out_w + kTX - 1) / kTX);
  return ctas <= 0x7fffffffLL;
}

}  // namespace

int resize_u8(const void* src, int B, int H, int W, int C, long long batch_stride, const int32_t* htab, int hk,
              const int32_t* vtab, int vk, void* out, int out_h, int out_w, cudaStream_t stream) {
  if (!src || !htab || !vtab || !out) return VT_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || C < 1 || C > 4 || hk < 1 || vk < 1 || out_h <= 0 || out_w <= 0) return VT_ERR_ARG;
  if (batch_stride < static_cast<long long>(H) * W * C) return VT_ERR_ARG;
  if (!grid_fits(out_h, out_w)) return VT_ERR_UNSUPPORTED;
  ResizeParams p = {};
  p.src = static_cast<const uint8_t*>(src);
  p.batch_stride = batch_stride;
  p.htab = htab;
  p.vtab = vtab;
  p.H = H; p.W = W; p.hk = hk; p.vk = vk;
  p.out = static_cast<uint8_t*>(out);
  p.out_h = out_h; p.out_w = out_w;
  return launch_resize_c<false>(p, C, B, stream);
}

int resize_u8_list(const vt_resize_image* images, int n_images, int C, const int32_t* tables, void* out, int out_h,
                   int out_w, cudaStream_t stream) {
  if (!images || !tables || !out) return VT_ERR_ARG;
  if (n_images <= 0 || C < 1 || C > 4 || out_h <= 0 || out_w <= 0) return VT_ERR_ARG;
  if (!grid_fits(out_h, out_w)) return VT_ERR_UNSUPPORTED;
  ResizeParams p = {};
  p.images = images;
  p.tables = tables;
  p.out = static_cast<uint8_t*>(out);
  p.out_h = out_h; p.out_w = out_w;
  return launch_resize_c<true>(p, C, n_images, stream);
}

}  // namespace vt

extern "C" int vt_resize_u8(const void* src, int32_t B, int32_t H, int32_t W, int32_t C, int64_t batch_stride,
                            const int32_t* htab, int32_t hk, const int32_t* vtab, int32_t vk, void* out,
                            int32_t out_h, int32_t out_w, void* stream) {
  return vt::resize_u8(src, B, H, W, C, batch_stride, htab, hk, vtab, vk, out, out_h, out_w,
                       static_cast<cudaStream_t>(stream));
}

extern "C" int vt_resize_u8_list(const vt_resize_image* images, int32_t n_images, int32_t C, const int32_t* tables,
                                 void* out, int32_t out_h, int32_t out_w, void* stream) {
  return vt::resize_u8_list(images, n_images, C, tables, out, out_h, out_w, static_cast<cudaStream_t>(stream));
}
