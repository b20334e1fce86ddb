/*
 * vitb200_clip.h — what libvitb200.so adds for CLIP image encoders (HF CLIPVisionModel, openai/clip-vit-*,
 * laion/CLIP-ViT-*): the activation codes of the GEMM epilogues, and a LayerNorm that also writes the row statistics of
 * its output.
 *
 * CLIP's MLP uses hidden_act="quick_gelu", x * sigmoid(1.702 x), in the OpenAI checkpoints.  The `act` argument of
 * vt_bgemm and the `gelu` argument of vt_gemm_bf16, vt_gemm_bf16_ln, vt_gemm_fp8 and vt_gemm_strided (vitb200.h) take
 * these codes.  vt_bgemm accepts all four; the other four accept VT_ACT_NONE, VT_ACT_GELU and VT_ACT_QUICK_GELU, and
 * return VT_ERR_ARG for any other value before anything is launched.  bf16 outputs of quick GELU are within one bf16
 * ulp of the correctly rounded x * sigmoid(1.702 x); fp32 outputs within 2e-6 relative + 1e-7 absolute.
 *
 * CLIP normalises the embeddings (pre_layrnorm) before the first block, so the residual stream starts as LN(embeddings)
 * and the statistics the first block's folded layernorm_before needs are those of the LayerNorm's output:
 * vt_layernorm_stats writes them in the same launch.
 *
 * Same conventions as vitb200.h (device pointers, dtype codes, void* stream, 0 / negative vt_status / positive
 * cudaError_t, no synchronisation, no device allocation, safe inside CUDA-graph capture), and exported from the same
 * library.
 */
#ifndef VITB200_CLIP_H_
#define VITB200_CLIP_H_

#include "vitb200.h"

#define VT_ACT_NONE 0
#define VT_ACT_GELU 1       /* exact-erf GELU, HF hidden_act="gelu" */
#define VT_ACT_TANH 2       /* tanh (vt_bgemm only: HF ViTPooler) */
#define VT_ACT_QUICK_GELU 3 /* x * sigmoid(1.702 x), HF hidden_act="quick_gelu" (CLIP) */

#ifdef __cplusplus
extern "C" {
#endif

/* vt_layernorm on bf16 rows (bf16 out, gamma / beta bf16 [dim]) that also writes the (sum, M2 = sum of squares about the
 * group's mean) of every 128-column group of every OUTPUT row, computed from the bf16 values it stores, to
 * stats[(row*(dim/128) + group)*2 .. +1] — the rowstats layout of vt_gemm_bf16_ln.  Row strides in elements
 * (multiples of 8), 16-byte aligned x / gamma / beta / out, 8-byte aligned stats; no atomics (bit-reproducible).  The
 * normalised output is the same bits as vt_layernorm's on the same rows.  dim % 128 != 0 returns VT_ERR_ARG,
 * dim > 1280 VT_ERR_UNSUPPORTED.  Replaces HF CLIPVisionTransformer.pre_layrnorm
 * (transformers/models/clip/modeling_clip.py) and the statistics the first block's folded layernorm_before reads. */
int vt_layernorm_stats(const void* x, const void* gamma, const void* beta, void* out, float* stats, int64_t rows,
                       int32_t dim, int64_t in_row_stride, int64_t out_row_stride, float eps, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* VITB200_CLIP_H_ */
