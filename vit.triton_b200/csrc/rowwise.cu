// Bandwidth-bound kernels: LayerNorm (K4), elementwise add (K5), row softmax (K6), CLS pooling (K7).
// All are vectorised (16-byte accesses), coalesced and warp-reduced; none uses shared memory
// because no element is touched by more than one thread.
//
// Reference semantics reproduced:
//   layernorm  vit/kernels/layernorm.py:51-85  (mean; biased variance of centred values;
//              w*(x-mean)/sqrt(var+eps)+b)
//   add        vit/kernels/add.py:60-65
//   softmax    vit/kernels/softmax.py:26-31    (max-subtracted exp / sum over the last dim)
#include "common.cuh"

namespace vt {

namespace {

template <typename T>
struct Vec;  // 16-byte vector of T

template <>
struct Vec<float> {
  static constexpr int N = 4;
  float v[4];
  __device__ __forceinline__ void load(const float* p) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  __device__ __forceinline__ void store(float* p) const {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};

template <>
struct Vec<__nv_bfloat16> {
  static constexpr int N = 8;
  float v[8];
  __device__ __forceinline__ void load(const __nv_bfloat16* p) {
    const uint4 t = *reinterpret_cast<const uint4*>(p);
    v[0] = bf16_lo(t.x); v[1] = bf16_hi(t.x);
    v[2] = bf16_lo(t.y); v[3] = bf16_hi(t.y);
    v[4] = bf16_lo(t.z); v[5] = bf16_hi(t.z);
    v[6] = bf16_lo(t.w); v[7] = bf16_hi(t.w);
  }
  __device__ __forceinline__ void store(__nv_bfloat16* p) const {
    uint4 t;
    t.x = pack_bf16x2(v[0], v[1]);
    t.y = pack_bf16x2(v[2], v[3]);
    t.z = pack_bf16x2(v[4], v[5]);
    t.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(p) = t;
  }
};

__device__ __forceinline__ float to_f(float x) { return x; }
__device__ __forceinline__ float to_f(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ void from_f(float* p, float x) { *p = x; }
__device__ __forceinline__ void from_f(__nv_bfloat16* p, float x) { *p = __float2bfloat16_rn(x); }

// ------------------------------------------------------------------------------------------
// LayerNorm: one warp per row, the row lives in registers (VPL 16-byte vectors per lane), so HBM
// sees exactly one read and one write of the activation.
// ------------------------------------------------------------------------------------------
template <typename T, typename TO, int VPL>
__global__ void __launch_bounds__(256)
layernorm_rows_kernel(const T* __restrict__ x, const T* __restrict__ gamma,
                      const T* __restrict__ beta, TO* __restrict__ out, long long rows, int dim,
                      long long in_stride, long long out_stride, float eps, int reverse) {
  constexpr int EV = Vec<T>::N;
  const int lane = threadIdx.x & 31;
  long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  if (reverse) row = rows - 1 - row;   // blocks are scheduled in index order: last rows first
  const T* xr = x + row * in_stride;
  const int nvec = dim / EV;

  Vec<T> d[VPL];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int vi = lane + i * 32;
    if (vi < nvec) {
      d[i].load(xr + vi * EV);
#pragma unroll
      for (int e = 0; e < EV; ++e) sum += d[i].v[e];
    }
  }
  const float mean0 = warp_sum(sum) / static_cast<float>(dim);
  float sq = 0.f, sc = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int vi = lane + i * 32;
    if (vi < nvec) {
#pragma unroll
      for (int e = 0; e < EV; ++e) {
        const float c = d[i].v[e] - mean0;
        sc += c;
        sq += c * c;
      }
    }
  }
  // sum / dim of fp32 values is not exact: the centred sum corrects it, so that a row of one repeated value gives
  // x - mean = 0 exactly (beta) instead of beta + gamma * (rounding residue) * rstd
  const float mean = mean0 + warp_sum(sc) / static_cast<float>(dim);
  const float var = warp_sum(sq) / static_cast<float>(dim);
  const float rstd = 1.0f / sqrtf(var + eps);

  TO* orow = out + row * out_stride;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int vi = lane + i * 32;
    if (vi < nvec) {
      Vec<T> g, b;
      g.load(gamma + vi * EV);
      b.load(beta + vi * EV);
      if constexpr (sizeof(TO) == sizeof(T)) {
        Vec<TO> o;
#pragma unroll
        for (int e = 0; e < EV; ++e) o.v[e] = g.v[e] * ((d[i].v[e] - mean) * rstd) + b.v[e];
        o.store(orow + vi * EV);
      } else {
        // fp32 in, bf16 out: 4 values -> 8 bytes
        static_assert(EV == 4, "mixed LN is fp32 -> bf16 only");
        uint2 o;
        o.x = pack_bf16x2(g.v[0] * ((d[i].v[0] - mean) * rstd) + b.v[0],
                          g.v[1] * ((d[i].v[1] - mean) * rstd) + b.v[1]);
        o.y = pack_bf16x2(g.v[2] * ((d[i].v[2] - mean) * rstd) + b.v[2],
                          g.v[3] * ((d[i].v[3] - mean) * rstd) + b.v[3]);
        *reinterpret_cast<uint2*>(orow + vi * EV) = o;
      }
    }
  }
}

// bf16 rows kept PACKED in registers (VPL x 4 registers instead of VPL x 8 unpacked floats) and
// unpacked in each of the three passes: <= 32 registers per thread, i.e. 64 resident warps per SM
// instead of 40 for layernorm_rows_kernel.  Same formula; the sums run over even / odd elements
// separately (packed pairs), so the last bit can differ from layernorm_rows_kernel.
// STATS (vt_layernorm_stats, dim % 128 == 0): also writes the (sum, M2 about the group mean) of every 128-column group of
// every OUTPUT row, computed from the bf16 values stored, to stats[(row * dim/128 + group) * 2 .. +1] — the rowstats
// layout of vt_gemm_bf16_ln.  A group is the 16 vectors of one half-warp, reduced in a fixed shuffle order (no
// atomics: bit-reproducible); the normalised output is the same arithmetic, so the same bits, as without STATS.  The
// statistics keep the stored row in registers: up to 64 per thread (4 blocks per SM) instead of 32, which spill.
template <int VPL, bool STATS = false>
__global__ void __launch_bounds__(256, STATS ? 4 : 8)
layernorm_bf16_packed_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ gamma,
                             const __nv_bfloat16* __restrict__ beta, __nv_bfloat16* __restrict__ out,
                             long long rows, int dim, long long in_stride, long long out_stride, float eps,
                             int reverse, float* __restrict__ stats = nullptr) {
  const int lane = threadIdx.x & 31;
  long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  if (reverse) row = rows - 1 - row;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * in_stride);
  const int nvec = dim >> 3;
  uint4 d[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int vi = lane + i * 32;
    d[i] = (vi < nvec) ? xr[vi] : make_uint4(0u, 0u, 0u, 0u);
  }
  // all arithmetic on packed fp32 pairs (FFMA2, sm_100 f32x2): the kernel is bound by instruction issue
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
  uint4* orow = reinterpret_cast<uint4*>(out + row * out_stride);
  const uint4* gp = reinterpret_cast<const uint4*>(gamma);
  const uint4* bp = reinterpret_cast<const uint4*>(beta);
  auto nrm = [&](uint32_t v, uint32_t g, uint32_t b) {
    const float2 t = __fmul2_rn(__fadd2_rn(up(v), nmean), rstd2);
    const float2 o = __ffma2_rn(up(g), t, up(b));
    return pack_bf16x2(o.x, o.y);
  };
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int vi = lane + i * 32;
    if (vi < nvec) {
      const uint4 g = __ldg(gp + vi);
      const uint4 b = __ldg(bp + vi);
      uint4 o;
      o.x = nrm(d[i].x, g.x, b.x);
      o.y = nrm(d[i].y, g.y, b.y);
      o.z = nrm(d[i].z, g.z, b.z);
      o.w = nrm(d[i].w, g.w, b.w);
      orow[vi] = o;
      if constexpr (STATS) d[i] = o;    // keep the stored bf16 values for the statistics
    }
  }
  if constexpr (STATS) {
    // dim % 128 == 0: a half-warp's 16 vectors (one group) are all valid or all past the row; the shuffles run on every
    // lane, invalid ones contributing zeros
    auto half_sum = [](float v) {
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      return v;
    };
    const int parts = dim >> 7;
    float2* srow = reinterpret_cast<float2*>(stats) + row * parts;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const bool valid = lane + i * 32 < nvec;
      float2 s = make_float2(0.f, 0.f);
      if (valid) {
        s = __fadd2_rn(up(d[i].x), up(d[i].y));
        s = __fadd2_rn(s, __fadd2_rn(up(d[i].z), up(d[i].w)));
      }
      const float sum = half_sum(s.x + s.y);
      const float2 ng = make_float2(-sum * (1.0f / 128.0f), -sum * (1.0f / 128.0f));
      float2 q = make_float2(0.f, 0.f);
      if (valid) {
        auto sq = [&](uint32_t w) { const float2 c = __fadd2_rn(up(w), ng); q = __ffma2_rn(c, c, q); };
        sq(d[i].x); sq(d[i].y); sq(d[i].z); sq(d[i].w);
      }
      const float m2 = half_sum(q.x + q.y);
      if (valid && (lane & 15) == 0) srow[2 * i + (lane >> 4)] = make_float2(sum, m2);
    }
  }
}

// Generic fallback (any dim / alignment): one warp per row, three passes over L1/L2-resident data.
template <typename T, typename TO>
__global__ void __launch_bounds__(256)
layernorm_generic_kernel(const T* __restrict__ x, const T* __restrict__ gamma,
                         const T* __restrict__ beta, TO* __restrict__ out, long long rows, int dim,
                         long long in_stride, long long out_stride, float eps) {
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const T* xr = x + row * in_stride;
  float sum = 0.f;
  for (int i = lane; i < dim; i += 32) sum += to_f(xr[i]);
  const float mean0 = warp_sum(sum) / static_cast<float>(dim);
  float sq = 0.f, sc = 0.f;
  for (int i = lane; i < dim; i += 32) {
    const float c = to_f(xr[i]) - mean0;
    sc += c;
    sq += c * c;
  }
  const float mean = mean0 + warp_sum(sc) / static_cast<float>(dim);   // as in layernorm_rows_kernel
  const float rstd = 1.0f / sqrtf(warp_sum(sq) / static_cast<float>(dim) + eps);
  TO* orow = out + row * out_stride;
  for (int i = lane; i < dim; i += 32)
    from_f(orow + i, to_f(gamma[i]) * ((to_f(xr[i]) - mean) * rstd) + to_f(beta[i]));
}

template <typename T, typename TO>
int launch_layernorm(const void* x, const void* g, const void* b, void* out, long long rows,
                     int dim, long long in_stride, long long out_stride, float eps, int reverse,
                     cudaStream_t stream) {
  constexpr int EV = Vec<T>::N;
  const int warps = 8;
  const unsigned grid = static_cast<unsigned>((rows + warps - 1) / warps);
  const T* xp = static_cast<const T*>(x);
  const T* gp = static_cast<const T*>(g);
  const T* bp = static_cast<const T*>(b);
  TO* op = static_cast<TO*>(out);
  const bool aligned =
      (dim % EV == 0) && (in_stride % EV == 0) && (out_stride % EV == 0) &&
      ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(g) |
        reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(out)) % 16 == 0);
  const int vpl = aligned ? (dim / EV + 31) / 32 : 0;
#ifndef VT_LN_UNPACKED   // default: packed-register kernel (30.1 vs 31.0 us per call at C2); -DVT_LN_UNPACKED for A/B runs
  if constexpr (sizeof(T) == 2 && sizeof(TO) == 2) {
    if (aligned && vpl >= 1 && vpl <= 5) {
#define VT_LNP_CASE(V)                                                                           \
  case V:                                                                                        \
    layernorm_bf16_packed_kernel<V><<<grid, warps * 32, 0, stream>>>(xp, gp, bp, op, rows, dim,  \
                                                                     in_stride, out_stride, eps, reverse); \
    break;
      switch (vpl) { VT_LNP_CASE(1) VT_LNP_CASE(2) VT_LNP_CASE(3) VT_LNP_CASE(4) VT_LNP_CASE(5) }
#undef VT_LNP_CASE
      return static_cast<int>(cudaGetLastError());
    }
  }
#endif
#define VT_LN_CASE(V)                                                                        \
  case V:                                                                                    \
    layernorm_rows_kernel<T, TO, V><<<grid, warps * 32, 0, stream>>>(xp, gp, bp, op, rows, dim, \
                                                                     in_stride, out_stride, eps, \
                                                                     reverse);                   \
    break;
  switch (vpl) {
    VT_LN_CASE(1) VT_LN_CASE(2) VT_LN_CASE(3) VT_LN_CASE(4) VT_LN_CASE(5) VT_LN_CASE(6)
    VT_LN_CASE(7) VT_LN_CASE(8) VT_LN_CASE(10) VT_LN_CASE(12) VT_LN_CASE(16)
    default:
      layernorm_generic_kernel<T, TO><<<grid, warps * 32, 0, stream>>>(xp, gp, bp, op, rows, dim,
                                                                       in_stride, out_stride, eps);
  }
#undef VT_LN_CASE
  return static_cast<int>(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------
// add: out = a + b, 16-byte vectors, 4 independent loads in flight per thread
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
add_vec_kernel(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ out,
               long long nvec) {
  constexpr int EV = Vec<T>::N;
  constexpr int U = 4;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  for (; i + (U - 1) * stride < nvec; i += U * stride) {
    Vec<T> va[U], vb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      va[u].load(a + (i + u * stride) * EV);
      vb[u].load(b + (i + u * stride) * EV);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
#pragma unroll
      for (int e = 0; e < EV; ++e) va[u].v[e] += vb[u].v[e];
      va[u].store(out + (i + u * stride) * EV);
    }
  }
  for (; i < nvec; i += stride) {
    Vec<T> va, vb;
    va.load(a + i * EV);
    vb.load(b + i * EV);
#pragma unroll
    for (int e = 0; e < EV; ++e) va.v[e] += vb.v[e];
    va.store(out + i * EV);
  }
}

template <typename T>
__global__ void add_scalar_kernel(const T* __restrict__ a, const T* __restrict__ b,
                                  T* __restrict__ out, long long start, long long n) {
  const long long i = start + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) from_f(out + i, to_f(a[i]) + to_f(b[i]));
}

template <typename T>
int launch_add(const void* a, const void* b, void* out, long long n, cudaStream_t stream) {
  constexpr int EV = Vec<T>::N;
  const T* ap = static_cast<const T*>(a);
  const T* bp = static_cast<const T*>(b);
  T* op = static_cast<T*>(out);
  const bool aligned = ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) |
                         reinterpret_cast<uintptr_t>(out)) % 16 == 0);
  long long done = 0;
  if (aligned && n >= EV) {
    const long long nvec = n / EV;
    long long blocks = (nvec + 256 * 4 - 1) / (256 * 4);
    const long long cap = 148LL * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    add_vec_kernel<T><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(ap, bp, op, nvec);
    done = nvec * EV;
  }
  if (done < n) {
    const long long rem = n - done;
    add_scalar_kernel<T><<<static_cast<unsigned>((rem + 255) / 256), 256, 0, stream>>>(ap, bp, op,
                                                                                      done, n);
  }
  return static_cast<int>(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------
// softmax over the last dim: one warp per row
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
softmax_rows_kernel(const T* __restrict__ x, T* __restrict__ out, long long rows, int cols,
                    long long row_stride) {
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const T* xr = x + row * row_stride;
  T* orow = out + row * static_cast<long long>(cols);
  float m = -INFINITY;
  for (int i = lane; i < cols; i += 32) m = fmaxf(m, to_f(xr[i]));
  m = warp_max(m);
  float s = 0.f;
  for (int i = lane; i < cols; i += 32) s += expf(to_f(xr[i]) - m);
  s = warp_sum(s);
  const float inv = 1.0f / s;
  for (int i = lane; i < cols; i += 32) from_f(orow + i, expf(to_f(xr[i]) - m) * inv);
}

// ------------------------------------------------------------------------------------------
// pool: out[b, :] = x[b, 0, :]  (CLS row of the final hidden states)
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void pool_cls_kernel(const T* __restrict__ x, T* __restrict__ out, int batch, int dim,
                                long long batch_stride) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(batch) * dim) return;
  const int b = static_cast<int>(i / dim);
  const int c = static_cast<int>(i - static_cast<long long>(b) * dim);
  out[i] = x[b * batch_stride + c];
}

// ------------------------------------------------------------------------------------------
// pool + all-gather over peer memory (K7): every rank stores the CLS rows of its images straight into
// the gather buffer of every peer (NVLink P2P stores, 16 bytes per thread), then raises a counter in
// that peer's flag array; the gathered rows are complete on a rank once every peer's counter in its own
// flag array shows the step, and are then copied into a plain local output buffer.  One kernel, no
// NCCL call: the transfer is 393 KB per rank at C2, i.e. latency-bound, and the kernel saves the
// separate pool launch, the NCCL launch and its internal synchronisation.
//
// Protocol (step e = 1, 2, ...; flags are monotonic counters, never reset; ALL state is in device memory
// — ctrl[0] = steps completed, ctrl[1] = block ticket — so a launch has no per-step argument and can be
// captured into a CUDA graph and replayed):
//   PUT  block (p, j) of rank r: e = ctrl[0] + 1; copy its slice of rows into peer p's buffer (e mod 4),
//        __syncthreads, thread 0: fence.sys + red.release.sys.add  flags_p[r] += 1.
//        The last block of the launch to finish (ticket) sets ctrl[0] = e.
//   GET  block (p, j): e = ctrl[0] - lag; thread 0 spins (ld.acquire.sys) until
//        flags_self[p] >= e * blocks_per_peer, then the block copies peer p's rows out of this rank's own
//        buffer (e mod 4) into the local output.
// PUT and GET are phases of ONE launch (mode PUT|GET: e is the step being put, the classic synchronous
// all-gather) or two launches: PUT of step i followed by GET with lag = 1 collects step i - 1, whose
// flags have long arrived, so no rank ever waits for a slower peer inside a step (the per-step barrier
// is off the critical path); GET with lag = 0 drains the last step.
// FOUR gather buffers are used in turn (e mod 4).  A peer can write step s into this rank's buffer once
// its own GET of step s - 1 (synchronous mode) or s - 2 (lag 1) is done, i.e. once this rank has finished
// PUT s - 1 / s - 2; this rank may then still have the GET of s - 1 (synchronous) or of s - 3 and s - 2
// (lag 1: GET s - 3 directly follows PUT s - 2 in the stream) in front of it — steps s - 3 .. s are the
// ones that can be live at once, anything older has been read.
// ------------------------------------------------------------------------------------------
constexpr int kMaxPeers = 16;
struct PeerTable {
  void* out[4][kMaxPeers];         // gather buffers of every rank, by step mod 4: (world * batch, dim) each
  unsigned int* flags[kMaxPeers];  // flag array of every rank, [world] counters
};
enum : int { PG_PUT = 1, PG_GET = 2 };

__global__ void __launch_bounds__(512)
pool_cls_allgather_kernel(const uint4* __restrict__ x, long long batch_stride_v, int batch, int dim_v,
                          const __grid_constant__ PeerTable peers, int rank, int world, int blocks_per_peer,
                          unsigned int* __restrict__ ctrl, uint4* __restrict__ out_local, int mode, unsigned int lag) {
  const int p = blockIdx.x / blocks_per_peer;      // peer this block talks to
  const int j = blockIdx.x - p * blocks_per_peer;
  const long long n = static_cast<long long>(batch) * dim_v;
  unsigned int done;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(done) : "l"(ctrl) : "memory");
  const unsigned int e = (mode & PG_PUT) ? done + 1u : done - lag;

  if (mode & PG_PUT) {
    uint4* dst = static_cast<uint4*>(peers.out[e & 3u][p]) + static_cast<long long>(rank) * n;
    for (long long i = static_cast<long long>(j) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<long long>(blocks_per_peer) * blockDim.x) {
      const int b = static_cast<int>(i / dim_v);
      const int c = static_cast<int>(i - static_cast<long long>(b) * dim_v);
      dst[i] = x[b * batch_stride_v + c];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence_system();
      asm volatile("red.release.sys.global.add.u32 [%0], 1;" ::"l"(peers.flags[p] + rank) : "memory");
    }
  }

  if ((mode & PG_GET) && static_cast<int>(e) > 0) {
    if (threadIdx.x == 0) {
      const unsigned int target = e * static_cast<unsigned int>(blocks_per_peer);
      const unsigned int* mine = peers.flags[rank] + p;
      unsigned long long t0;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
      unsigned int v;
      for (;;) {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
        if (static_cast<int>(v - target) >= 0) break;
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (now - t0 > 120000000000ULL) {   // 120 s: a peer died; surface it as a CUDA error, not a hang
          printf("vt: pool_cls_allgather timeout rank %d waiting for rank %d (flag %u, want %u)\n", rank, p, v,
                 target);
          __trap();
        }
        __nanosleep(64);
      }
    }
    __syncthreads();
    // peer p's rows have landed in this rank's buffer (written over NVLink: read them from L2, not L1)
    const uint4* src = static_cast<const uint4*>(peers.out[e & 3u][rank]) + static_cast<long long>(p) * n;
    uint4* dst = out_local + static_cast<long long>(p) * n;
    for (long long i = static_cast<long long>(j) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<long long>(blocks_per_peer) * blockDim.x)
      dst[i] = __ldcg(src + i);
  }

  if (mode & PG_PUT) {
    // every block has read ctrl[0] before it takes a ticket, so the last ticket may advance the step
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned int ticket = atomicAdd(ctrl + 1, 1u);
      if (ticket == gridDim.x - 1) {
        ctrl[1] = 0u;
        __threadfence();
        asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(ctrl), "r"(e) : "memory");
      }
    }
  }
}

}  // namespace

int pool_cls_allgather(const void* x, int batch, int dim, long long batch_stride, int dtype,
                       void* const* peer_out, unsigned int* const* peer_flags, int rank, int world,
                       unsigned int* ctrl, void* out_local, int mode, int lag, cudaStream_t stream) {
  if (!peer_out || !peer_flags || !ctrl || batch <= 0 || dim <= 0 || world <= 0 || world > kMaxPeers ||
      rank < 0 || rank >= world || (mode & ~(PG_PUT | PG_GET)) || mode == 0 || lag < 0)
    return VT_ERR_ARG;
  if ((mode & PG_PUT) && (!x || lag != 0)) return VT_ERR_ARG;
  if ((mode & PG_GET) && !out_local) return VT_ERR_ARG;
  const int es = dtype == VT_F32 ? 4 : dtype == VT_BF16 ? 2 : 0;
  if (es == 0) return VT_ERR_DTYPE;
  const int per16 = 16 / es;
  if ((dim % per16) || (batch_stride % per16) || (reinterpret_cast<uintptr_t>(x) & 15) ||
      (reinterpret_cast<uintptr_t>(out_local) & 15) || (reinterpret_cast<uintptr_t>(ctrl) & 7))
    return VT_ERR_ALIGN;
  PeerTable t;
  for (int p = 0; p < world; ++p) {
    if (!peer_flags[p]) return VT_ERR_ARG;
    for (int b = 0; b < 4; ++b) {
      void* o = peer_out[b * world + p];
      if (!o || (reinterpret_cast<uintptr_t>(o) & 15)) return VT_ERR_ARG;
      t.out[b][p] = o;
    }
    t.flags[p] = peer_flags[p];
  }
  const int dim_v = dim / per16;
  const long long n = static_cast<long long>(batch) * dim_v;
  int blocks_per_peer = static_cast<int>((n + 512 * 8 - 1) / (512 * 8));   // ~8 vectors per thread
  if (blocks_per_peer < 1) blocks_per_peer = 1;
  if (blocks_per_peer > 8) blocks_per_peer = 8;
  pool_cls_allgather_kernel<<<world * blocks_per_peer, 512, 0, stream>>>(
      static_cast<const uint4*>(x), batch_stride / per16, batch, dim_v, t, rank, world, blocks_per_peer, ctrl,
      static_cast<uint4*>(out_local), mode, static_cast<unsigned int>(lag));
  return static_cast<int>(cudaGetLastError());
}

int layernorm_rows(const void* x, const void* gamma, const void* beta, void* out, long long rows,
                   int dim, long long in_stride, long long out_stride, float eps, int in_dtype,
                   int out_dtype, int reverse, cudaStream_t stream) {
  if (!x || !gamma || !beta || !out || rows < 0 || dim <= 0) return VT_ERR_ARG;
  if (rows == 0) return VT_OK;
  if (in_dtype == VT_F32 && out_dtype == VT_F32)
    return launch_layernorm<float, float>(x, gamma, beta, out, rows, dim, in_stride, out_stride,
                                          eps, reverse, stream);
  if (in_dtype == VT_BF16 && out_dtype == VT_BF16)
    return launch_layernorm<__nv_bfloat16, __nv_bfloat16>(x, gamma, beta, out, rows, dim,
                                                          in_stride, out_stride, eps, reverse, stream);
  if (in_dtype == VT_F32 && out_dtype == VT_BF16)
    return launch_layernorm<float, __nv_bfloat16>(x, gamma, beta, out, rows, dim, in_stride,
                                                  out_stride, eps, reverse, stream);
  return VT_ERR_DTYPE;
}

// vt_layernorm_stats: the packed kernel vt_layernorm runs for these rows (bf16, dim <= 1280, 16-byte aligned) with the
// row statistics of its output written as well.
int layernorm_stats(const void* x, const void* gamma, const void* beta, void* out, float* stats, long long rows, int dim,
                    long long in_stride, long long out_stride, float eps, int reverse, cudaStream_t stream) {
  if (!x || !gamma || !beta || !out || !stats || rows < 0 || dim <= 0 || (dim % 128)) return VT_ERR_ARG;
  if (dim > 5 * 32 * 8) return VT_ERR_UNSUPPORTED;
  if ((in_stride % 8) || (out_stride % 8) ||
      ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta) |
        reinterpret_cast<uintptr_t>(out)) & 15) || (reinterpret_cast<uintptr_t>(stats) & 7))
    return VT_ERR_ALIGN;
  if (rows == 0) return VT_OK;
  const int warps = 8;
  const unsigned grid = static_cast<unsigned>((rows + warps - 1) / warps);
  const auto* xp = static_cast<const __nv_bfloat16*>(x);
  const auto* gp = static_cast<const __nv_bfloat16*>(gamma);
  const auto* bp = static_cast<const __nv_bfloat16*>(beta);
  auto* op = static_cast<__nv_bfloat16*>(out);
#define VT_LNS_CASE(V)                                                                                               \
  case V:                                                                                                            \
    layernorm_bf16_packed_kernel<V, true><<<grid, warps * 32, 0, stream>>>(xp, gp, bp, op, rows, dim, in_stride,     \
                                                                           out_stride, eps, reverse, stats);         \
    break;
  switch ((dim / 8 + 31) / 32) { VT_LNS_CASE(1) VT_LNS_CASE(2) VT_LNS_CASE(3) VT_LNS_CASE(4) VT_LNS_CASE(5) }
#undef VT_LNS_CASE
  return static_cast<int>(cudaGetLastError());
}

int add_elementwise(const void* a, const void* b, void* out, long long n, int dtype,
                    cudaStream_t stream) {
  if (!a || !b || !out || n < 0) return VT_ERR_ARG;
  if (n == 0) return VT_OK;
  if (dtype == VT_F32) return launch_add<float>(a, b, out, n, stream);
  if (dtype == VT_BF16) return launch_add<__nv_bfloat16>(a, b, out, n, stream);
  return VT_ERR_DTYPE;
}

int softmax_rows(const void* x, void* out, long long rows, int cols, long long row_stride,
                 int dtype, cudaStream_t stream) {
  if (!x || !out || rows < 0 || cols <= 0) return VT_ERR_ARG;
  if (rows == 0) return VT_OK;
  const unsigned grid = static_cast<unsigned>((rows + 7) / 8);
  if (dtype == VT_F32)
    softmax_rows_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(x),
                                                         static_cast<float*>(out), rows, cols,
                                                         row_stride);
  else if (dtype == VT_BF16)
    softmax_rows_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(
        static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(out), rows, cols,
        row_stride);
  else
    return VT_ERR_DTYPE;
  return static_cast<int>(cudaGetLastError());
}

int pool_cls(const void* x, void* out, int batch, int dim, long long batch_stride, int dtype,
             cudaStream_t stream) {
  if (!x || !out || batch < 0 || dim <= 0) return VT_ERR_ARG;
  if (batch == 0) return VT_OK;
  const long long n = static_cast<long long>(batch) * dim;
  const unsigned grid = static_cast<unsigned>((n + 255) / 256);
  if (dtype == VT_F32)
    pool_cls_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(x),
                                                     static_cast<float*>(out), batch, dim,
                                                     batch_stride);
  else if (dtype == VT_BF16)
    pool_cls_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(
        static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(out), batch, dim,
        batch_stride);
  else
    return VT_ERR_DTYPE;
  return static_cast<int>(cudaGetLastError());
}

// Row gather (vt_gather_rows): out[i, :] = x[idx[i], :] — the CLS rows of a ragged batch, whose images start at
// arbitrary packed rows.  One block per output row, element copies (a few hundred rows per call).
template <typename T>
__global__ void __launch_bounds__(256)
gather_rows_kernel(const T* __restrict__ x, long long ldx, const long long* __restrict__ idx, T* __restrict__ out,
                   long long ldo, int cols) {
  const long long src = __ldg(idx + blockIdx.x);
  const T* in = x + src * ldx;
  T* o = out + static_cast<long long>(blockIdx.x) * ldo;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) o[c] = in[c];
}

int gather_rows(const void* x, long long ldx, const long long* idx, void* out, long long ldo, int rows, int cols,
                int dtype, cudaStream_t stream) {
  if (!x || !idx || !out || rows < 0 || cols <= 0 || ldx < cols || ldo < cols) return VT_ERR_ARG;
  if (rows == 0) return VT_OK;
  if (dtype == VT_F32)
    gather_rows_kernel<float><<<rows, 256, 0, stream>>>(static_cast<const float*>(x), ldx, idx,
                                                        static_cast<float*>(out), ldo, cols);
  else if (dtype == VT_BF16)
    gather_rows_kernel<__nv_bfloat16><<<rows, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(x), ldx, idx,
                                                                static_cast<__nv_bfloat16*>(out), ldo, cols);
  else
    return VT_ERR_DTYPE;
  return static_cast<int>(cudaGetLastError());
}

}  // namespace vt
