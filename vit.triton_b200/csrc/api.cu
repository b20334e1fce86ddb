// extern "C" surface of libvitb200.so (declared in include/vitb200.h and its companions
// vitb200_resolution.h, vitb200_ragged.h, vitb200_mask.h, vitb200_tokens.h, vitb200_clip.h).  Thin: argument plumbing
// only, all kernels live in the other translation units.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/vitb200.h"
#include "../../include/vitb200_resolution.h"
#include "../../include/vitb200_ragged.h"
#include "../../include/vitb200_mask.h"
#include "../../include/vitb200_tokens.h"
#include "../../include/vitb200_clip.h"

namespace vt {
int layernorm_rows(const void*, const void*, const void*, void*, long long, int, long long,
                   long long, float, int, int, int, cudaStream_t);
int layernorm_stats(const void*, const void*, const void*, void*, float*, long long, int, long long, long long, float, int,
                    cudaStream_t);
int add_elementwise(const void*, const void*, void*, long long, int, cudaStream_t);
int softmax_rows(const void*, void*, long long, int, long long, int, cudaStream_t);
int pool_cls(const void*, void*, int, int, long long, int, cudaStream_t);
int pool_cls_allgather(const void*, int, int, long long, int, void* const*, unsigned int* const*, int, int,
                       unsigned int*, void*, int, int, cudaStream_t);
int gemm_bf16_tcgen05(const void*, long long, const void*, long long, void*, long long, int,
                      const float*, const void*, long long, int, int, int, int, cudaStream_t);
int gemm2_bf16_tcgen05(const void*, long long, const void*, long long, void*, long long, const float*,
                       const void*, long long, int, int, int, int, const float*, const float*, int, float,
                       float*, int, cudaStream_t);
void gemm2_set_debug_buffer(void*);
void attn5_set_debug_buffer(void*);
void attn5_set_bound(int);
void attn5_set_max_ctas(int);
void gemm2_set_max_groups(int);
int simt_gemm(const void*, const void*, void*, const void*, int, int, int, int, int,
              const long long*, const long long*, const long long*, float, int, int, cudaStream_t);
int attn5_fwd_tcgen05(const void*, const void*, const void*, void*, int, int, int, int, long long,
                      long long, long long, long long, float, int, cudaStream_t);
int attn5mb_fwd_tcgen05(const void*, const void*, const void*, void*, int, int, int, int, long long,
                        long long, long long, long long, float, int, cudaStream_t);
int patching(const void*, void*, int, int, int, int, int, int, cudaStream_t);
int bgemm_tcgen05(const void*, const void*, void*, const float*, const void*, int, int, int, int, int, const long long*,
                  const long long*, const long long*, int, float, int, int, cudaStream_t);
int pack_bf16(const void*, int, void*, int, int, int, int, const long long*, const long long*, int, int, int,
              cudaStream_t);
int gemm2_fp8_tcgen05(const void*, long long, const void*, long long, void*, long long, int, const float*, const float*,
                      const void*, long long, int, int, int, int, float, int, cudaStream_t);
int layernorm_e4m3(const void*, const void*, const void*, void*, long long, int, long long, long long, float, float,
                   cudaStream_t);
int quantize_rows_e4m3(const void*, long long, void*, long long, float*, int, int, cudaStream_t);
int patch_gather(const void*, int, void*, int, int, int, int, int, int, int, int, cudaStream_t);
int pos_resample(const void*, int, float*, int, int, int, int, int, cudaStream_t);
int patch_gather_ragged(const void*, int, int, int, int, void*, long long, void*, int, long long, int, cudaStream_t);
int gather_rows(const void*, long long, const long long*, void*, long long, int, int, int, cudaStream_t);
int gemm2_patch_tokens(const void*, long long, const void*, long long, void*, const float*, const void*, float*, int, int,
                       int, int, int, int, cudaStream_t);
int ln_fold(const void*, long long, const float*, const float*, const float*, void*, long long, float*, float*, int,
            int, int, cudaStream_t);
int embed_finalize(void*, const void*, const void*, int, int, int, int, int, cudaStream_t);
int patch_gather_masked(const void*, int, const void*, const void*, const void*, void*, long long, void*, int, int, int,
                        int, int, int, int, cudaStream_t);
int embed_finalize_masked(void*, const void*, const void*, const void*, const void*, int, int, int, int, int,
                          cudaStream_t);
int mim_reconstruct(const void*, void*, int, int, int, int, int, int, const void*, int, const float*, float, const void*,
                    float*, float*, cudaStream_t);
int conv2d_nchw(const void*, const void*, const void*, void*, int, int, int, int, int, int, int,
                int, cudaStream_t);
}  // namespace vt

static inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }

// Traversal direction of the hot-path kernels.  In the forward every kernel consumes what the
// previous launch produced; both walk their rows in index order, so by the time the consumer
// starts, the producer's FIRST rows have long been evicted from L2 while its LAST rows are still
// resident.  Consecutive launches therefore alternate direction (row tiles / work items from the
// end): the consumer starts on the rows the producer wrote last.  Results do not depend on the
// direction; VT_TRAVERSAL=0 disables the alternation (A/B measurements).
static int next_direction() {
  static const bool enabled = [] {
    const char* e = getenv("VT_TRAVERSAL");
    return !(e && e[0] == '0');
  }();
  static thread_local int parity = 0;
  const int d = parity;
  parity ^= 1;
  return enabled ? d : 0;
}

extern "C" {

int vt_version(void) { return 100; }

// Developer hook (not part of the public header): per-CTA cycle counters of the 2-CTA GEMM.
void vt_debug_set_buffer(void* ptr) { vt::gemm2_set_debug_buffer(ptr); }
void vt_debug_set_attn_buffer(void* ptr) {
  vt::attn5_set_debug_buffer(ptr);
}
// Developer hook: 0 = every attention item takes the exact two-pass softmax, 1 = items whose logits are bounded
// skip the row-max pass (the default), -1 = back to the VT_ATTN_NO_BOUND environment default.
void vt_debug_set_attn_bound(int mode) { vt::attn5_set_bound(mode); }
// Developer hook (SM partitioning experiments): the 2-CTA GEMM launches at most `gemm_groups` groups of four CTAs and the
// single-block attention kernel at most `attn_ctas` CTAs; 0 = all SMs.  Read at launch time (also during graph capture).
void vt_debug_set_sm_partition(int gemm_groups, int attn_ctas) {
  vt::gemm2_set_max_groups(gemm_groups);
  vt::attn5_set_max_ctas(attn_ctas);
}

const char* vt_status_string(int status) {
  switch (status) {
    case VT_OK: return "ok";
    case VT_ERR_ARG: return "invalid argument (null pointer or bad shape)";
    case VT_ERR_DTYPE: return "unsupported dtype";
    case VT_ERR_ALIGN: return "pointer/stride alignment not met for the tensor-core path";
    case VT_ERR_UNSUPPORTED: return "shape not supported by this kernel";
    case VT_ERR_DRIVER: return "cuTensorMapEncodeTiled unavailable or failed";
    default:
      if (status > 0) return cudaGetErrorString(static_cast<cudaError_t>(status));
      return "unknown status";
  }
}

int vt_layernorm(const void* x, const void* gamma, const void* beta, void* out, int64_t rows,
                 int32_t dim, int64_t in_row_stride, int64_t out_row_stride, float eps,
                 int32_t in_dtype, int32_t out_dtype, void* stream) {
  return vt::layernorm_rows(x, gamma, beta, out, rows, dim, in_row_stride, out_row_stride, eps,
                            in_dtype, out_dtype, next_direction(), S(stream));
}

int vt_layernorm_stats(const void* x, const void* gamma, const void* beta, void* out, float* stats, int64_t rows,
                       int32_t dim, int64_t in_row_stride, int64_t out_row_stride, float eps, void* stream) {
  return vt::layernorm_stats(x, gamma, beta, out, stats, rows, dim, in_row_stride, out_row_stride, eps,
                             next_direction(), S(stream));
}

int vt_add(const void* a, const void* b, void* out, int64_t n, int32_t dtype, void* stream) {
  return vt::add_elementwise(a, b, out, n, dtype, S(stream));
}

int vt_softmax(const void* x, void* out, int64_t rows, int32_t cols, int64_t in_row_stride,
               int32_t dtype, void* stream) {
  return vt::softmax_rows(x, out, rows, cols, in_row_stride, dtype, S(stream));
}

int vt_gemm_bf16(const void* A, int64_t lda, const void* Bt, int64_t ldb, void* out, int64_t ldo,
                 int32_t out_dtype, const float* bias, const void* residual, int64_t ldr,
                 int32_t M, int32_t N, int32_t K, int32_t gelu, void* stream) {
  // bf16 output -> 2-CTA kernel (gemm2_sm100.cu); fp32 output -> 1-CTA kernel (gemm_sm100.cu).
  // VT_GEMM_IMPL=1 forces the 1-CTA kernel (A/B measurements only).
  static const int impl = [] {
    const char* e = getenv("VT_GEMM_IMPL");
    return (e && e[0] == '1') ? 1 : 2;
  }();
  if (out_dtype == VT_BF16 && impl == 2)
    return vt::gemm2_bf16_tcgen05(A, lda, Bt, ldb, out, ldo, bias, residual, ldr, M, N, K, gelu, nullptr,
                                  nullptr, 0, 0.f, nullptr, next_direction(), S(stream));
  return vt::gemm_bf16_tcgen05(A, lda, Bt, ldb, out, ldo, out_dtype, bias, residual, ldr, M, N, K,
                               gelu, S(stream));
}

int vt_gemm_bf16_ln(const void* A, int64_t lda, const void* Bt, int64_t ldb, void* out, int64_t ldo,
                    const float* bias, const void* residual, int64_t ldr, int32_t M, int32_t N, int32_t K,
                    int32_t gelu, const float* rowstats, const float* colsum, int32_t ln_dim, float ln_eps,
                    float* stats_out, void* stream) {
  return vt::gemm2_bf16_tcgen05(A, lda, Bt, ldb, out, ldo, bias, residual, ldr, M, N, K, gelu, rowstats,
                                colsum, ln_dim, ln_eps, stats_out, next_direction(), S(stream));
}

int vt_gemm_strided(const void* A, const void* B, void* C, const void* bias, int32_t M, int32_t N,
                    int32_t K, int32_t batch_outer, int32_t batch_inner, const int64_t* sA,
                    const int64_t* sB, const int64_t* sC, float scale, int32_t gelu, int32_t dtype,
                    void* stream) {
  if (!sA || !sB || !sC) return VT_ERR_ARG;
  long long a[4], b[4], c[4];
  for (int i = 0; i < 4; ++i) { a[i] = sA[i]; b[i] = sB[i]; c[i] = sC[i]; }
  return vt::simt_gemm(A, B, C, bias, M, N, K, batch_outer, batch_inner, a, b, c, scale, gelu,
                       dtype, S(stream));
}

int vt_gemm_fp8(const void* A, int64_t lda, const void* Bt, int64_t ldb, void* out, int64_t ldo, int32_t out_dtype,
                const float* bias, const float* colscale, const void* residual, int64_t ldr, int32_t M, int32_t N,
                int32_t K, int32_t gelu, float out_scale, void* stream) {
  if (out_dtype != VT_BF16 && out_dtype != VT_E4M3) return VT_ERR_DTYPE;
  return vt::gemm2_fp8_tcgen05(A, lda, Bt, ldb, out, ldo, out_dtype == VT_E4M3, bias, colscale, residual, ldr, M, N, K,
                               gelu, out_scale, next_direction(), S(stream));
}

int vt_layernorm_fp8(const void* x, const void* gamma, const void* beta, void* out, int64_t rows, int32_t dim,
                     int64_t in_row_stride, int64_t out_row_stride, float eps, float out_scale, void* stream) {
  return vt::layernorm_e4m3(x, gamma, beta, out, rows, dim, in_row_stride, out_row_stride, eps, out_scale, S(stream));
}

int vt_quantize_rows_fp8(const void* w, int64_t ldw, void* out, int64_t ldo, float* scales, int32_t N, int32_t K,
                         void* stream) {
  return vt::quantize_rows_e4m3(w, ldw, out, ldo, scales, N, K, S(stream));
}

int vt_bgemm(const void* A, const void* B, void* C, const float* bias, const void* residual, int32_t M, int32_t N,
             int32_t K, int32_t batch_outer, int32_t batch_inner, const int64_t* sA, const int64_t* sB, const int64_t* sC,
             int32_t b_mn_major, float scale, int32_t act, int32_t out_dtype, void* stream) {
  if (!sA || !sB || !sC) return VT_ERR_ARG;
  long long a[3], b[3], c[3];
  for (int i = 0; i < 3; ++i) { a[i] = sA[i]; b[i] = sB[i]; c[i] = sC[i]; }
  return vt::bgemm_tcgen05(A, B, C, bias, residual, M, N, K, batch_outer, batch_inner, a, b, c, b_mn_major, scale, act,
                           out_dtype, S(stream));
}

int vt_pack_bf16(const void* src, int32_t src_dtype, void* dst, int32_t rows, int32_t cols, int32_t batch_outer,
                 int32_t batch_inner, const int64_t* s_src, const int64_t* s_dst, int32_t cpad, int32_t pieces,
                 int32_t pattern, void* stream) {
  if (!s_src || !s_dst) return VT_ERR_ARG;
  long long a[4], d[3];
  for (int i = 0; i < 4; ++i) a[i] = s_src[i];
  for (int i = 0; i < 3; ++i) d[i] = s_dst[i];
  return vt::pack_bf16(src, src_dtype, dst, rows, cols, batch_outer, batch_inner, a, d, cpad, pieces, pattern, S(stream));
}

int vt_flash_attn(const void* q, const void* k, const void* v, void* out, int32_t B, int32_t H,
                  int32_t N, int32_t dh, int64_t qkv_row_stride, int64_t qkv_batch_stride,
                  int64_t out_row_stride, int64_t out_batch_stride, float scale, void* stream) {
  // Persistent two-group kernels (csrc/attn5_sm100.cu): the single-block kernel for head dim 64 and
  // N <= 208, the online-softmax multi-block kernel for longer sequences and for head dim 80 (ViT-H).
  // Anything else returns VT_ERR_UNSUPPORTED and the host shim takes the exact strided path.
  if (dh == 64 && N <= 208)
    return vt::attn5_fwd_tcgen05(q, k, v, out, B, H, N, dh, qkv_row_stride, qkv_batch_stride,
                                 out_row_stride, out_batch_stride, scale, next_direction(), S(stream));
  if (dh == 64 || dh == 80)
    return vt::attn5mb_fwd_tcgen05(q, k, v, out, B, H, N, dh, qkv_row_stride, qkv_batch_stride,
                                   out_row_stride, out_batch_stride, scale, next_direction(), S(stream));
  return VT_ERR_UNSUPPORTED;
}

int vt_ln_fold(const void* w, int64_t ldw, const float* bias, const float* gamma, const float* beta, void* w_out,
               int64_t ldo, float* bias_out, float* colsum_out, int32_t N, int32_t K, int32_t zero_sum, void* stream) {
  return vt::ln_fold(w, ldw, bias, gamma, beta, w_out, ldo, bias_out, colsum_out, N, K, zero_sum, S(stream));
}

int vt_patch_embed_gemm(const void* pixels, int32_t pix_dtype, const void* w, int64_t ldw, const float* bias,
                        const void* posb, void* out, float* stats_out, void* workspace, int32_t B, int32_t C, int32_t S_,
                        int32_t P, int32_t D, void* stream) {
  if (P <= 0 || S_ <= 0 || (S_ % P)) return VT_ERR_ARG;
  return vt_patch_embed_gemm_hw(pixels, pix_dtype, w, ldw, bias, posb, out, stats_out, workspace, B, C, S_, S_, P, D,
                                stream);
}

int vt_patch_embed_gemm_hw(const void* pixels, int32_t pix_dtype, const void* w, int64_t ldw, const float* bias,
                           const void* posb, void* out, float* stats_out, void* workspace, int32_t B, int32_t C,
                           int32_t H, int32_t W, int32_t P, int32_t D, void* stream) {
  return vt_patch_embed_gemm_hw_prefix(pixels, pix_dtype, w, ldw, bias, posb, out, stats_out, workspace, B, C, H, W, P,
                                       D, 1, stream);
}

int vt_patch_embed_gemm_hw_prefix(const void* pixels, int32_t pix_dtype, const void* w, int64_t ldw, const float* bias,
                                  const void* posb, void* out, float* stats_out, void* workspace, int32_t B, int32_t C,
                                  int32_t H, int32_t W, int32_t P, int32_t D, int32_t prefix, void* stream) {
  if (P <= 0 || H < P || W < P || !workspace || prefix < 1 || prefix > 2) return VT_ERR_ARG;
  const long long n = static_cast<long long>(H / P) * (W / P);
  if (n + 32 > 0x7fffffffLL) return VT_ERR_UNSUPPORTED;
  const int tokens = static_cast<int>(n) + prefix;
  const int tok_pad = (tokens + 31) & ~31;
  const int K = C * P * P;
  if (ldw < K || (ldw % 8)) return VT_ERR_ALIGN;
  const int rc = vt::patch_gather(pixels, pix_dtype, workspace, B, C, H, W, P, tok_pad, static_cast<int>(ldw), prefix,
                                  S(stream));
  if (rc) return rc;
  return vt::gemm2_patch_tokens(workspace, ldw, w, ldw, out, bias, posb, stats_out, B, tok_pad, tokens, D,
                                static_cast<int>(ldw), next_direction(), S(stream));
}

int vt_pos_embed_resample(const void* pos, int32_t pos_dtype, float* out, int32_t D, int32_t g_in, int32_t gh,
                          int32_t gw, void* stream) {
  return vt_pos_embed_resample_prefix(pos, pos_dtype, out, D, g_in, gh, gw, 1, stream);
}

int vt_pos_embed_resample_prefix(const void* pos, int32_t pos_dtype, float* out, int32_t D, int32_t g_in, int32_t gh,
                                 int32_t gw, int32_t prefix, void* stream) {
  return vt::pos_resample(pos, pos_dtype, out, D, g_in, gh, gw, prefix, S(stream));
}

int vt_patch_embed_ragged_gather(const vt_ragged_image* images, int32_t n_images, int32_t pix_dtype, int32_t C,
                                 int32_t P, void* patches, int64_t ldw, void* table, int32_t D, int64_t M,
                                 void* stream) {
  return vt_patch_embed_ragged_gather_prefix(images, n_images, pix_dtype, C, P, patches, ldw, table, D, M, 1, stream);
}

int vt_patch_embed_ragged_gather_prefix(const vt_ragged_image* images, int32_t n_images, int32_t pix_dtype, int32_t C,
                                        int32_t P, void* patches, int64_t ldw, void* table, int32_t D, int64_t M,
                                        int32_t prefix, void* stream) {
  return vt::patch_gather_ragged(images, n_images, pix_dtype, C, P, patches, ldw, table, D, M, prefix, S(stream));
}

int vt_gather_rows(const void* x, int64_t ldx, const int64_t* idx, void* out, int64_t ldo, int32_t rows, int32_t cols,
                   int32_t dtype, void* stream) {
  return vt::gather_rows(x, ldx, reinterpret_cast<const long long*>(idx), out, ldo, rows, cols, dtype, S(stream));
}

int vt_patching(const void* image, void* out, int32_t B, int32_t C, int32_t H, int32_t W, int32_t P,
                int32_t dtype, void* stream) {
  return vt::patching(image, out, B, C, H, W, P, dtype, S(stream));
}

int vt_embed_finalize(void* x, const void* pos, const void* cls, int32_t B, int32_t N, int32_t D,
                      int32_t dtype, void* stream) {
  return vt_embed_finalize_prefix(x, pos, cls, B, N, D, dtype, 1, stream);
}

int vt_embed_finalize_prefix(void* x, const void* pos, const void* prefix_rows, int32_t B, int32_t N, int32_t D,
                             int32_t dtype, int32_t prefix, void* stream) {
  return vt::embed_finalize(x, pos, prefix_rows, B, N, D, dtype, prefix, S(stream));
}

int vt_patch_embed_masked_gather(const void* pixels, int32_t pix_dtype, const void* mask, const void* pos,
                                 const void* posm, void* patches, int64_t ldw, void* table, int32_t B, int32_t C,
                                 int32_t H, int32_t W, int32_t P, int32_t D, void* stream) {
  return vt_patch_embed_masked_gather_prefix(pixels, pix_dtype, mask, pos, posm, patches, ldw, table, B, C, H, W, P, D,
                                             1, stream);
}

int vt_patch_embed_masked_gather_prefix(const void* pixels, int32_t pix_dtype, const void* mask, const void* pos,
                                        const void* posm, void* patches, int64_t ldw, void* table, int32_t B,
                                        int32_t C, int32_t H, int32_t W, int32_t P, int32_t D, int32_t prefix,
                                        void* stream) {
  return vt::patch_gather_masked(pixels, pix_dtype, mask, pos, posm, patches, ldw, table, B, C, H, W, P, D, prefix,
                                 S(stream));
}

int vt_embed_finalize_masked(void* x, const void* pos, const void* cls, const void* mask_token, const void* mask,
                             int32_t B, int32_t N, int32_t D, int32_t dtype, void* stream) {
  return vt_embed_finalize_masked_prefix(x, pos, cls, mask_token, mask, B, N, D, dtype, 1, stream);
}

int vt_embed_finalize_masked_prefix(void* x, const void* pos, const void* prefix_rows, const void* mask_token,
                                    const void* mask, int32_t B, int32_t N, int32_t D, int32_t dtype, int32_t prefix,
                                    void* stream) {
  return vt::embed_finalize_masked(x, pos, prefix_rows, mask_token, mask, B, N, D, dtype, prefix, S(stream));
}

int vt_mim_reconstruct(const void* dec, void* rec, int32_t dtype, int32_t B, int32_t C, int32_t gh, int32_t gw,
                       int32_t s, const void* pixels, int32_t pix_dtype, const float* norm, float rescale,
                       const void* mask, float* partial, float* loss, void* stream) {
  return vt::mim_reconstruct(dec, rec, dtype, B, C, gh, gw, s, pixels, pix_dtype, norm, rescale, mask, partial, loss,
                             S(stream));
}

int vt_conv2d(const void* input, const void* weight, const void* bias, void* out, int32_t B,
              int32_t C, int32_t H, int32_t W, int32_t O, int32_t kh, int32_t kw, int32_t dtype,
              void* stream) {
  return vt::conv2d_nchw(input, weight, bias, out, B, C, H, W, O, kh, kw, dtype, S(stream));
}

int vt_pool_cls(const void* x, void* out, int32_t B, int32_t D, int64_t batch_stride, int32_t dtype,
                void* stream) {
  return vt::pool_cls(x, out, B, D, batch_stride, dtype, S(stream));
}

int vt_pool_cls_allgather(const void* x, int32_t B, int32_t D, int64_t batch_stride, int32_t dtype,
                          void* const* peer_out, uint32_t* const* peer_flags, int32_t rank, int32_t world,
                          uint32_t* ctrl, void* out_local, int32_t mode, int32_t lag, void* stream) {
  return vt::pool_cls_allgather(x, B, D, batch_stride, dtype, peer_out,
                                reinterpret_cast<unsigned int* const*>(peer_flags), rank, world,
                                reinterpret_cast<unsigned int*>(ctrl), out_local, mode, lag, S(stream));
}

}  // extern "C"
