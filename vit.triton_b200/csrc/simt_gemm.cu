// Generic strided batched GEMM on the FP32 SIMT pipe.
//
// This is the exact-fp32 and odd-shape path behind the `matmul` / `matmul3` entry points
// (reference vit/kernels/matmul.py:111-156, matmul3.py:111-156): arbitrary strides, any M/N/K,
// fp32 or bf16 storage, fp32 accumulation, optional bias / exact-erf or quick GELU / scale epilogue.
// The bf16 model path never comes here for its dense layers (those run on tcgen05, see
// gemm_sm100.cu); the fp32 parity configuration (C1, <=1e-3 vs HF) does, because single-pass
// TF32 tensor-core math misses that tolerance (SURVEY.md 7.2).
#include "common.cuh"

namespace vt {

namespace {

constexpr int TM = 64, TN = 64, TK = 16;

struct SimtGemmParams {
  const void* A;
  const void* B;
  void* C;
  const void* bias;   // dtype of C... stored as T (same as inputs) or null
  int M, N, K;
  int batch_inner;    // z = zo * batch_inner + zi
  long long sAo, sAi, sAm, sAk;
  long long sBo, sBi, sBk, sBn;
  long long sCo, sCi, sCm, sCn;
  float scale;
  int gelu;
};

__device__ __forceinline__ float ldf(const float* p) { return *p; }
__device__ __forceinline__ float ldf(const __nv_bfloat16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void stf(float* p, float v) { *p = v; }
__device__ __forceinline__ void stf(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

template <typename T>
__global__ void __launch_bounds__(256)
simt_gemm_kernel(const SimtGemmParams p) {
  __shared__ float As[TK][TM + 4];
  __shared__ float Bs[TK][TN + 4];

  const int z = blockIdx.z;
  const int zo = z / p.batch_inner;
  const int zi = z - zo * p.batch_inner;
  const T* A = static_cast<const T*>(p.A) + zo * p.sAo + zi * p.sAi;
  const T* B = static_cast<const T*>(p.B) + zo * p.sBo + zi * p.sBi;
  T* C = static_cast<T*>(p.C) + zo * p.sCo + zi * p.sCi;

  const int m0 = blockIdx.y * TM;
  const int n0 = blockIdx.x * TN;
  const int tid = threadIdx.x;
  const int tx = tid & 15;   // column group
  const int ty = tid >> 4;   // row group

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  // Loader mapping: choose the thread-fastest index along the contiguous memory direction.
  const bool a_k_contig = (p.sAk == 1);
  const bool b_n_contig = (p.sBn == 1);

  for (int k0 = 0; k0 < p.K; k0 += TK) {
#pragma unroll
    for (int it = 0; it < (TM * TK) / 256; ++it) {
      const int idx = tid + it * 256;
      int m, k;
      if (a_k_contig) { k = idx % TK; m = idx / TK; } else { m = idx % TM; k = idx / TM; }
      const int gm = m0 + m, gk = k0 + k;
      As[k][m] = (gm < p.M && gk < p.K) ? ldf(A + gm * p.sAm + gk * p.sAk) : 0.f;
    }
#pragma unroll
    for (int it = 0; it < (TN * TK) / 256; ++it) {
      const int idx = tid + it * 256;
      int n, k;
      if (b_n_contig) { n = idx % TN; k = idx / TN; } else { k = idx % TK; n = idx / TK; }
      const int gn = n0 + n, gk = k0 + k;
      Bs[k][n] = (gn < p.N && gk < p.K) ? ldf(B + gk * p.sBk + gn * p.sBn) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
      const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

  const T* bias = static_cast<const T*>(p.bias);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      if (gn >= p.N) continue;
      float v = acc[i][j];
      if (bias) v += ldf(bias + gn);
      if (p.gelu == kActGelu) v = gelu_erf(v);
      else if (p.gelu == kActQuickGelu) v = quick_gelu(v);
      v *= p.scale;
      stf(C + gm * p.sCm + gn * p.sCn, v);
    }
  }
}

}  // namespace

int simt_gemm(const void* A, const void* B, void* C, const void* bias, int M, int N, int K,
              int batch_outer, int batch_inner, const long long* sA, const long long* sB,
              const long long* sC, float scale, int gelu, int dtype, cudaStream_t stream) {
  if (!A || !B || !C || M < 0 || N < 0 || K < 0 || batch_outer < 0 || batch_inner <= 0 || !gemm_act_ok(gelu))
    return VT_ERR_ARG;
  if (M == 0 || N == 0 || batch_outer == 0) return VT_OK;
  const long long nz = static_cast<long long>(batch_outer) * batch_inner;
  if (nz > 65535) return VT_ERR_UNSUPPORTED;
  SimtGemmParams p;
  p.A = A; p.B = B; p.C = C; p.bias = bias;
  p.M = M; p.N = N; p.K = K;
  p.batch_inner = batch_inner;
  p.sAo = sA[0]; p.sAi = sA[1]; p.sAm = sA[2]; p.sAk = sA[3];
  p.sBo = sB[0]; p.sBi = sB[1]; p.sBk = sB[2]; p.sBn = sB[3];
  p.sCo = sC[0]; p.sCi = sC[1]; p.sCm = sC[2]; p.sCn = sC[3];
  p.scale = scale;
  p.gelu = gelu;
  dim3 grid((N + TN - 1) / TN, (M + TM - 1) / TM, static_cast<unsigned>(nz));
  if (grid.y > 65535) return VT_ERR_UNSUPPORTED;
  if (dtype == VT_F32)
    simt_gemm_kernel<float><<<grid, 256, 0, stream>>>(p);
  else if (dtype == VT_BF16)
    simt_gemm_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(p);
  else
    return VT_ERR_DTYPE;
  return static_cast<int>(cudaGetLastError());
}

}  // namespace vt
