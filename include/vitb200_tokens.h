/*
 * vitb200_tokens.h — entry points of libvitb200.so for models with more than one token in front of the patches:
 * DeiT (HF DeiTModel, facebook/deit-*-distilled-*) puts a learned distillation token after CLS, so its sequence is
 * [CLS, DIST, patch 0, ...], N = prefix + gh * gw tokens with prefix = 2, and its position table has prefix + g^2 rows.
 *
 * Each function is an existing entry point with one more argument, int32_t prefix, the number of tokens in front of
 * the patches: 1 (ViT: CLS) or 2 (DeiT: CLS, distillation token); any other value returns VT_ERR_ARG before anything is
 * launched.  Row t < prefix of an image is a prefix token; patch p is row prefix + p.  At prefix = 1 each one is the
 * function it generalises (which calls it with 1): same launches, same grids, same bits.
 *
 * Same conventions as vitb200.h (device pointers, dtype codes, void* stream, 0 / negative vt_status / positive
 * cudaError_t, no synchronisation, no device allocation, safe inside CUDA-graph capture), and exported from the same
 * library.  They are declared here rather than in the other headers so that their entry-point sets stay fixed.
 */
#ifndef VITB200_TOKENS_H_
#define VITB200_TOKENS_H_

#include "vitb200.h"
#include "vitb200_ragged.h"

#ifdef __cplusplus
extern "C" {
#endif

/* vt_patch_embed_gemm_hw with `prefix` leading tokens: tokens = prefix + gh*gw, workspace bf16
 * [B, roundup(tokens, 32), ldw] with rows t < prefix zero and patch p at row prefix + p; posb bf16 [tokens, D] with
 * row t < prefix = token_t + pos[t] - bias; out bf16 [B, tokens, D].  Replaces DeiTPatchEmbeddings.forward plus the
 * CLS / distillation / position add of DeiTEmbeddings.forward (transformers/models/deit/modeling_deit.py). */
int vt_patch_embed_gemm_hw_prefix(const void* pixels, int32_t pix_dtype, const void* w, int64_t ldw, const float* bias,
                                  const void* posb, void* out, float* stats_out, void* workspace, int32_t B, int32_t C,
                                  int32_t H, int32_t W, int32_t P, int32_t D, int32_t prefix, void* stream);

/* vt_patch_embed_masked_gather with `prefix` leading tokens: N = prefix + gh*gw rows per image; masked patch p is row
 * b * N + prefix + p (mask[b, p]); rows t < prefix are zero patches with table rows pos[t]. */
int vt_patch_embed_masked_gather_prefix(const void* pixels, int32_t pix_dtype, const void* mask, const void* pos,
                                        const void* posm, void* patches, int64_t ldw, void* table, int32_t B,
                                        int32_t C, int32_t H, int32_t W, int32_t P, int32_t D, int32_t prefix,
                                        void* stream);

/* vt_patch_embed_ragged_gather with `prefix` leading tokens per image: a descriptor's tokens must be
 * prefix + (height / P) * (width / P); patch p of an image is row row0 + prefix + p, rows row0 .. row0 + prefix - 1
 * are zero patches.  Every row of [0, M) is written once, and nothing outside it. */
int vt_patch_embed_ragged_gather_prefix(const vt_ragged_image* images, int32_t n_images, int32_t pix_dtype, int32_t C,
                                        int32_t P, void* patches, int64_t ldw, void* table, int32_t D, int64_t M,
                                        int32_t prefix, void* stream);

/* vt_pos_embed_resample with `prefix` leading rows: pos [prefix + g_in^2, D] -> out f32 [prefix + gh*gw, D]; rows
 * t < prefix are copied, the grid starting at row prefix is resampled.  Replaces
 * DeiTEmbeddings.interpolate_pos_encoding (transformers/models/deit/modeling_deit.py). */
int vt_pos_embed_resample_prefix(const void* pos, int32_t pos_dtype, float* out, int32_t D, int32_t g_in, int32_t gh,
                                 int32_t gw, int32_t prefix, void* stream);

/* vt_embed_finalize with `prefix` leading tokens: x [B, N, D] holds the patch projections in rows prefix .. N - 1;
 * x[b, t] = prefix_rows[t] + pos[t] for t < prefix, x[b, t] += pos[t] otherwise.  prefix_rows [prefix, D]
 * ([cls; distillation token]) and pos [N, D] in x's dtype; N >= prefix. */
int vt_embed_finalize_prefix(void* x, const void* pos, const void* prefix_rows, int32_t B, int32_t N, int32_t D,
                             int32_t dtype, int32_t prefix, void* stream);

/* vt_embed_finalize_masked with `prefix` leading tokens: mask [B, N - prefix]; x[b, t] = prefix_rows[t] + pos[t] for
 * t < prefix, (mask[b, t - prefix] ? mask_token : x[b, t]) + pos[t] otherwise. */
int vt_embed_finalize_masked_prefix(void* x, const void* pos, const void* prefix_rows, const void* mask_token,
                                    const void* mask, int32_t B, int32_t N, int32_t D, int32_t dtype, int32_t prefix,
                                    void* stream);

#ifdef __cplusplus
}
#endif

#endif /* VITB200_TOKENS_H_ */
