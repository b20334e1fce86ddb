/*
 * vitb200.h — C ABI of libvitb200.so: the sm_100a (B200) kernels behind the vit.triton host API.
 *
 * Every entry point
 *   - takes raw DEVICE pointers, integer sizes / element strides, a dtype enum and a cudaStream_t
 *     (passed as void*); no torch / C++ types cross the boundary;
 *   - enqueues work on the given stream and returns immediately (never synchronises, never
 *     allocates device memory, safe inside CUDA-graph capture);
 *   - returns 0 on success, a NEGATIVE vt_status for argument errors, or a POSITIVE cudaError_t.
 *
 * The reference (cmeraki/vit.triton) has no native boundary: its kernels are Triton functions
 * called from Python.  Each declaration below cites the reference Python entry point it replaces;
 * the Python shim in vit.triton_b200/vit/kernels/ keeps those names and signatures and calls this
 * ABI through ctypes (see INTEGRATION.md).
 */
#ifndef VITB200_H_
#define VITB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  VT_OK = 0,
  VT_ERR_ARG = -1,         /* bad shape / null pointer */
  VT_ERR_DTYPE = -2,       /* unsupported dtype */
  VT_ERR_ALIGN = -3,       /* pointer or stride alignment not met for the tensor-core path */
  VT_ERR_UNSUPPORTED = -4, /* shape outside what this kernel implements */
  VT_ERR_DRIVER = -5       /* cuTensorMapEncodeTiled unavailable / failed */
} vt_status;

typedef enum { VT_F32 = 0, VT_BF16 = 1, VT_U8 = 2 /* raw NHWC pixel inputs only */, VT_E4M3 = 3 /* FP8 path only */ } vt_dtype;

/* Library version (major*10000 + minor*100 + patch). */
int vt_version(void);

/* Human-readable text for a status returned by any function below (static storage). */
const char* vt_status_string(int status);

/* K4 — LayerNorm over the last dim of a [rows, dim] matrix; biased variance, eps inside sqrt.
 * Replaces layernorm_triton / LayerNormTriton.forward (vit/kernels/layernorm.py:90-127,129-142).
 * in/out dtype pairs: f32->f32, bf16->bf16, f32->bf16.  gamma/beta have the INPUT dtype. */
int vt_layernorm(const void* x, const void* gamma, const void* beta, void* out, int64_t rows,
                 int32_t dim, int64_t in_row_stride, int64_t out_row_stride, float eps,
                 int32_t in_dtype, int32_t out_dtype, void* stream);

/* K5 — out = a + b over n contiguous elements.  Replaces add_triton (vit/kernels/add.py:67-104). */
int vt_add(const void* a, const void* b, void* out, int64_t n, int32_t dtype, void* stream);

/* K6 — softmax over the last dim of [rows, cols] (input row stride in elements, output dense).
 * Replaces softmax_triton (vit/kernels/softmax.py:36-74). */
int vt_softmax(const void* x, void* out, int64_t rows, int32_t cols, int64_t in_row_stride,
               int32_t dtype, void* stream);

/* K1 — tensor-core GEMM (tcgen05 + TMEM + TMA):  out[M,N] = epi(A[M,K] . Bt[N,K]^T + bias).
 * A, Bt bf16, K-major (row strides lda / ldb in elements, multiples of 8; K, N multiples of 8).
 * out / residual: bf16 or f32 (out_dtype); bias: f32 or NULL; gelu: epilogue activation, VT_ACT_NONE /
 * VT_ACT_GELU (exact erf) / VT_ACT_QUICK_GELU of vitb200_clip.h (0 / 1 / 3; others: VT_ERR_ARG);
 * residual (nullable) is added after the bias and may alias out.
 * Replaces matmul_triton (vit/kernels/matmul.py:111-156) for the model's dense layers and folds
 * add_triton (vit/vit.py:140,147) into the epilogue. */
int vt_gemm_bf16(const void* A, int64_t lda, const void* Bt, int64_t ldb, void* out, int64_t ldo,
                 int32_t out_dtype, const float* bias, const void* residual, int64_t ldr,
                 int32_t M, int32_t N, int32_t K, int32_t gelu, void* stream);

/* K1 with LayerNorm folded into the epilogue and/or row statistics emitted for the next fold (bf16 out).
 *   rowstats != NULL (with colsum): A is the UN-normalised activation; row m's statistics are given as
 *     ln_dim/128 partial pairs rowstats[(m*(ln_dim/128) + i)*2 .. +1] = (sum, M2) of the i-th group of 128
 *     elements, M2 = sum of squares about the GROUP's mean; the groups are merged the Chan / Welford way
 *     (in index order: bit-reproducible), so the variance is a sum of centred squares like the reference's
 *     two-pass kernel (vit/kernels/layernorm.py:51-85) even for rows with |mean| >> std; a row whose
 *     variance is exactly 0 yields out = bias_n (= LN's beta through the dense layer).
 *     ln_dim % 128 == 0; Bt must carry gamma
 *     (Bt[n,k] = W[n,k] * gamma[k]), bias must carry beta (bias[n] + sum_k beta[k] W[n,k]) and
 *     colsum[n] = sum_k Bt[n,k]:   out = rstd_m * acc - rstd_m * mean_m * colsum_n + bias_n  (then the activation:
 *     gelu as for vt_gemm_bf16).
 *     colsum == NULL: the rows of Bt sum to zero (Bt[n,k] = W[n,k]*gamma[k] - mean_k(W[n,k]*gamma[k])), the
 *     mean term is then part of acc and   out = rstd_m * acc + bias_n.
 *   stats_out != NULL (needs residual, N % 128 == 0): writes the (sum, M2) of every 128-column group
 *     of every output row to stats_out[(m*(N/128) + group)*2 .. +1] — the rowstats layout above.
 * Replaces layernorm_triton (vit/kernels/layernorm.py:90-127) + matmul_triton for the
 * LN -> dense pairs of Transformer.forward (vit/vit.py:133-144). */
int vt_gemm_bf16_ln(const void* A, int64_t lda, const void* Bt, int64_t ldb, void* out, int64_t ldo,
                    const float* bias, const void* residual, int64_t ldr, int32_t M, int32_t N, int32_t K,
                    int32_t gelu, const float* rowstats, const float* colsum, int32_t ln_dim, float ln_eps,
                    float* stats_out, void* stream);

/* Pack-time fold of a LayerNorm (gamma, beta: f32 [K]) into the dense layer that consumes it, producing the
 * operands vt_gemm_bf16_ln expects.  w, w_out: bf16 [N, K] K-major (row strides ldw / ldo in elements);
 * bias (f32 [N], nullable) -> bias_out[n] = bias[n] + sum_k w[n,k] * beta[k].
 *   zero_sum == 0: w_out[n,k] = bf16(w[n,k] * gamma[k]), colsum_out[n] = sum_k w_out[n,k]  (f32 [N])
 *   zero_sum != 0: every row of w * gamma is shifted by its own mean before rounding and the rounding
 *     residue of the row sum is cancelled by re-rounding the elements nearest to a tie (each element moves
 *     by at most one bf16 ulp), so sum_k w_out[n,k] ~ 1e-6 and the GEMM needs no colsum; colsum_out may be
 *     NULL (when given it receives the remaining row sums).
 * Deterministic.  Replaces nothing in the reference (it has no fused LayerNorm); it is what lets
 * layernorm_triton (vit/kernels/layernorm.py:90-127) disappear into matmul_triton's epilogue. */
int vt_ln_fold(const void* w, int64_t ldw, const float* bias, const float* gamma, const float* beta, void* w_out,
               int64_t ldo, float* bias_out, float* colsum_out, int32_t N, int32_t K, int32_t zero_sum, void* stream);

/* Generic strided batched GEMM on the FP32 pipe (exact-fp32 path and odd shapes):
 *   C[z] = scale * act(A[z] . B[z] + bias),  z = zo * batch_inner + zi
 * strides (elements): sA = {outer, inner, m, k}, sB = {outer, inner, k, n}, sC = {outer, inner, m, n}.
 * All tensors share `dtype`; bias nullable; gelu: VT_ACT_NONE / VT_ACT_GELU / VT_ACT_QUICK_GELU (vitb200_clip.h).
 * Replaces matmul_triton (matmul.py:111-156) and matmul3's matmul_triton (matmul3.py:111-156)
 * wherever the tensor-core path's alignment rules do not hold. */
int vt_gemm_strided(const void* A, const void* B, void* C, const void* bias, int32_t M, int32_t N,
                    int32_t K, int32_t batch_outer, int32_t batch_inner, const int64_t* sA,
                    const int64_t* sB, const int64_t* sC, float scale, int32_t gelu, int32_t dtype,
                    void* stream);

/* Optional FP8 path (off the bf16 headline metric; SURVEY.md 8f-3) — K1 on tcgen05.mma kind::f8f6f4:
 *   out[M,N] = act( (A8[M,K] . B8[N,K]^T) * colscale[n] + bias[n] ) (+ residual)
 * A8, B8: e4m3 bytes, K-major, row strides lda / ldb in BYTES (multiples of 16, K % 16 == 0); colscale f32 [N] =
 * per-output-channel weight scale x activation scale; bias f32 [N] (nullable); residual bf16 (nullable, ldr in elements);
 * out_dtype VT_BF16 (ldo in elements) or VT_E4M3: out8 = e4m3(out * out_scale), ldo in bytes, N % 128 == 0, no residual;
 * gelu (act): VT_ACT_NONE / VT_ACT_GELU / VT_ACT_QUICK_GELU (vitb200_clip.h).
 * Replaces matmul_triton (vit/kernels/matmul.py:111-156) for the QKV / fc1 / fc2 layers when the FP8 path is on. */
int vt_gemm_fp8(const void* A, int64_t lda, const void* Bt, int64_t ldb, void* out, int64_t ldo, int32_t out_dtype,
                const float* bias, const float* colscale, const void* residual, int64_t ldr, int32_t M, int32_t N,
                int32_t K, int32_t gelu, float out_scale, void* stream);

/* K4 with the FP8 quantisation of the GEMM operand fused in: out8[m,:] = e4m3( LN(x[m,:]) * out_scale ), bf16 in
 * (x, gamma, beta), e4m3 bytes out (row strides in elements / bytes).  layernorm_triton
 * (vit/kernels/layernorm.py:90-127) for the FP8 path. */
int vt_layernorm_fp8(const void* x, const void* gamma, const void* beta, void* out, int64_t rows, int32_t dim,
                     int64_t in_row_stride, int64_t out_row_stride, float eps, float out_scale, void* stream);

/* Pack-time weight quantisation: w bf16 [N,K] (row stride ldw elements) -> out8[n,:] = e4m3(w[n,:] / scales[n]),
 * scales[n] = amax_k |w[n,k]| / 448 (1 for an all-zero row); ldo in bytes; K % 4 == 0. */
int vt_quantize_rows_fp8(const void* w, int64_t ldw, void* out, int64_t ldo, float* scales, int32_t N, int32_t K,
                         void* stream);

/* Batched general GEMM on the tensor cores (tcgen05 + TMEM + TMA, 4-D tensor maps):
 *   C[zo,zi] = act( scale * A[zo,zi] . B[zo,zi] + bias ) (+ residual[zo,zi]),  zo < batch_outer, zi < batch_inner
 * A: bf16 [M, K] per batch, K contiguous; element strides sA = {outer, inner, row}.
 * B: bf16; b_mn_major == 0: [N, K] per batch, K contiguous; != 0: [K, N] per batch, N contiguous (the layout
 *    matmul3 receives) — consumed in place as an MN-major UMMA operand; sB = {outer, inner, row}.
 *    A batch stride of 0 broadcasts the operand along that level (A and B alike); both batch strides 0 =
 *    one matrix shared by all batches (weights).
 * C / residual: out_dtype (bf16 | f32) [M, N] per batch, sC = {outer, inner, row}; bias f32 [N] (nullable);
 * act: VT_ACT_* of vitb200_clip.h: 0 none, 1 exact-erf GELU, 2 tanh, 3 quick GELU.  Any M, N, K; every A / B stride a multiple of 8 elements and
 * both bases 16-byte aligned (pack with vt_pack_bf16 otherwise).
 * Replaces matmul3's matmul_triton (vit/kernels/matmul3.py:111-156); with split fp32 operands
 * (vt_pack_bf16, pieces = 3) also matmul_triton (vit/kernels/matmul.py:111-156) for the fp32 model, whose
 * tl.dot (matmul.py:92) is a TF32 tensor-core product; with act = 2 the HF pooler dense + tanh the reference's
 * loader maps (vit/utils.py:63-64). */
int vt_bgemm(const void* A, const void* B, void* C, const float* bias, const void* residual, int32_t M, int32_t N,
             int32_t K, int32_t batch_outer, int32_t batch_inner, const int64_t* sA, const int64_t* sB, const int64_t* sC,
             int32_t b_mn_major, float scale, int32_t act, int32_t out_dtype, void* stream);

/* Operand packing for vt_bgemm: src (src_dtype f32 | bf16) [rows, cols] per batch with ANY element strides
 * s_src = {outer, inner, row, col} -> dst bf16 rows of pieces * cpad elements (s_dst = {outer, inner, row}),
 * columns cols .. cpad-1 of every piece zero.  pieces == 1: plain conversion (transpose / pad).
 * pieces == 3: x = hi + lo with hi = bf16(x), lo = bf16(x - hi), laid out [hi | hi | lo] (pattern 0, the A
 * operand) or [hi | lo | hi] (pattern 1, the B operand): one bf16 GEMM over K' = 3 * cpad then accumulates
 * a_hi b_hi + a_hi b_lo + a_lo b_hi in fp32 ("3 x bf16" fp32 product, ~2^-16 relative).
 * pieces == 6: three-way split x = x1 + x2 + x3, A side [a1|a1|a2|a1|a2|a3], B side [b1|b2|b1|b3|b2|b1]: the six
 * products of weight >= 2^-16 (no more accurate than 3 pieces on B200: the fp32 accumulator truncates). */
int vt_pack_bf16(const void* src, int32_t src_dtype, void* dst, int32_t rows, int32_t cols, int32_t batch_outer,
                 int32_t batch_inner, const int64_t* s_src, const int64_t* s_dst, int32_t cpad, int32_t pieces,
                 int32_t pattern, void* stream);

/* K3 — fused attention forward (tcgen05, flash style, no materialised scores), bf16:
 *   out[b, i, h*dh:(h+1)*dh] = softmax_j( scale * q[b,i,h] . k[b,j,h] ) v[b,j,h]
 * head dim 64 or 80, any N >= 1, scale > 0 and finite.
 * q/k/v: [B, N, H*dh] views with common row / batch strides (e.g. slices of a fused-QKV buffer, or three
 * allocations); out: [B, N, H*dh] with its own row / batch strides.  Every pointer 16-byte aligned, every stride a
 * multiple of 8 elements.  Nothing outside out's [B, N, H*dh] view is written, and nothing outside the q/k/v views
 * is read.
 * Returns VT_ERR_ARG for a null pointer or B, H, N <= 0; VT_ERR_ALIGN for a misaligned pointer or stride;
 * VT_ERR_UNSUPPORTED, before anything is launched, for another head dim, a scale that is not positive and finite
 * (the kernels take the row maximum of the raw scores), or a batch too large for one launch.
 * Replaces the per-head matmul3 -> softmax -> matmul3 -> slice-assign chain (vit/vit.py:60-72,101-108). */
int vt_flash_attn(const void* q, const void* k, const void* v, void* out, int32_t B, int32_t H,
                  int32_t N, int32_t dh, int64_t qkv_row_stride, int64_t qkv_batch_stride,
                  int64_t out_row_stride, int64_t out_batch_stride, float scale, void* stream);

/* K2 — patch embedding with CLS + position embedding fused, as two launches: a bandwidth-bound gather of the pixels
 * into padded bf16 patch rows — every pixel read once — followed by the 2-CTA tcgen05 GEMM in token mode, whose
 * epilogue adds the conv bias and the position table.
 * pixels [B,C,S,S] (pix_dtype f32|bf16) with w [D, C*P*P] bf16 in (c,i,j) order (row stride ldw), or
 * pixels [B,S,S,C] (pix_dtype VT_U8: raw NHWC bytes) with w in (i,j,c) order — the caller folds the image processor's
 * rescale / mean / std into w and bias (vit/packing.py:pack_embeddings); ldw >= C*P*P, multiple of 8: the K padding
 * of w must be zero.  bias f32 [D] = conv bias (uint8 pixels: minus the folded mean term); posb bf16 [n+1, D] =
 * position embeddings with row 0 = cls + pos[0] - bias; out bf16 [B, n+1, D]; workspace: bf16
 * [B, roundup(n+1, 32), ldw] scratch owned by the caller (the gathered patch rows).
 * stats_out != NULL (D % 128 == 0): also writes the (sum, M2 about the group mean) of every 128-column group of every
 * output row (CLS rows included) to stats_out[(row*(D/128) + group)*2 .. +1] — the rowstats layout of
 * vt_gemm_bf16_ln, so the first block's layernorm_before folds into its QKV GEMM too.
 * Replaces Conv2DTriton.forward + Embeddings.forward glue (conv2d.py:100-167, vit/vit.py:188-200); the uint8 form
 * also replaces the HF ViTImageProcessor rescale + normalise step in front of it. */
int vt_patch_embed_gemm(const void* pixels, int32_t pix_dtype, const void* w, int64_t ldw, const float* bias,
                        const void* posb, void* out, float* stats_out, void* workspace, int32_t B, int32_t C, int32_t S,
                        int32_t P, int32_t D, void* stream);

/* (B,C,H,W) -> (B, (H/P)*(W/P), C*P*P) patch rows in (c,i,j) order.
 * Replaces patching_triton (vit/kernels/patching.py:54-92). */
int vt_patching(const void* image, void* out, int32_t B, int32_t C, int32_t H, int32_t W, int32_t P,
                int32_t dtype, void* stream);

/* x[b,0,:] = cls + pos[0];  x[b,t,:] += pos[t] for t >= 1, in place on x [B,N,D].
 * Replaces torch.cat(cls) and the broadcast + position_embeddings (vit/vit.py:195-200). */
int vt_embed_finalize(void* x, const void* pos, const void* cls, int32_t B, int32_t N, int32_t D,
                      int32_t dtype, void* stream);

/* Stride == kernel convolution, NCHW in / NCHW out, any kernel shape.
 * Replaces conv2d_triton (vit/kernels/conv2d.py:100-150) as a standalone entry point. */
int vt_conv2d(const void* input, const void* weight, const void* bias, void* out, int32_t B,
              int32_t C, int32_t H, int32_t W, int32_t O, int32_t kh, int32_t kw, int32_t dtype,
              void* stream);

/* K7 — out[b,:] = x[b,0,:]: CLS rows of the final hidden states, the tensor the data-parallel
 * wrapper all-gathers.  (New: the reference has no pooling / multi-GPU step.) */
int vt_pool_cls(const void* x, void* out, int32_t B, int32_t D, int64_t batch_stride, int32_t dtype,
                void* stream);

/* K7 fused with its collective — pool + all-gather over peer memory in ONE kernel (no NCCL call).
 * Rank `rank` stores the CLS rows of its B images into rows [rank*B, (rank+1)*B) of every peer's gather
 * buffer and raises the counter peer_flags[p][rank] (PUT); the gathered (world*B, D) rows are copied from
 * this rank's own gather buffer into out_local once peer_flags[rank][p] of every p shows the step (GET).
 *   peer_out    HOST array of 4*world device pointers: [b*world + p] = gather buffer b (0..3) of rank p,
 *               (world*B, D) each, P2P-mapped (e.g. torch symmetric memory); step e uses buffer e mod 4
 *   peer_flags  HOST array of `world` device pointers to uint32[world] counters, zeroed once before step 1
 *   ctrl        this rank's uint32[2] in device memory, zeroed once: [0] = steps completed, [1] = scratch.
 *               The step number lives THERE, not in an argument: launches are identical from step to step
 *               and can be captured into a CUDA graph.
 *   mode        VT_PG_PUT | VT_PG_GET: synchronous all-gather of this step (returns once every peer's rows of
 *               this step are in out_local); VT_PG_PUT: store + signal only, never waits; VT_PG_GET: collect
 *               step (steps completed - lag) — after a PUT, lag 1 collects the PREVIOUS step (no rank waits
 *               for a slower peer inside a step), lag 0 drains the last one.  x is ignored for GET alone,
 *               out_local for PUT alone.
 * All ranks must pass the same B, D, dtype and issue the same sequence of modes.  world <= 16.  A peer that
 * never arrives traps the kernel after 120 s.
 * (New: the reference has no multi-GPU step; replaces vt_pool_cls + ncclAllGather.) */
#define VT_PG_PUT 1
#define VT_PG_GET 2
int vt_pool_cls_allgather(const void* x, int32_t B, int32_t D, int64_t batch_stride, int32_t dtype,
                          void* const* peer_out, uint32_t* const* peer_flags, int32_t rank, int32_t world,
                          uint32_t* ctrl, void* out_local, int32_t mode, int32_t lag, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* VITB200_H_ */
