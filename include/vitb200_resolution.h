/*
 * vitb200_resolution.h — entry points of libvitb200.so that run a checkpoint at an input resolution other than the
 * one its position table was trained for, square or not (HF ViTModel's interpolate_pos_encoding=True).
 *
 * Same conventions as vitb200.h (device pointers, dtype codes, void* stream, 0 / negative vt_status / positive
 * cudaError_t, no synchronisation, no device allocation, safe inside CUDA-graph capture), and exported from the same
 * library.  They are declared here rather than in vitb200.h so that the core header's entry-point set stays fixed.
 * The reference (cmeraki/vit.triton) has no interpolation; each declaration cites the HF function it replaces.
 */
#ifndef VITB200_RESOLUTION_H_
#define VITB200_RESOLUTION_H_

#include "vitb200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* vt_patch_embed_gemm with a rectangular input: pixels [B,C,H,W] (pix_dtype f32|bf16) or [B,H,W,C] (VT_U8).  The patch
 * grid is gh x gw = (H / P) x (W / P) rounded down: the last H % P rows and W % P columns are dropped, as HF's stride-P
 * Conv2d drops them.  posb bf16 [1 + gh*gw, D] (row 0 = cls + pos[0] - bias), out bf16 [B, 1 + gh*gw, D], workspace
 * bf16 [B, roundup(1 + gh*gw, 32), ldw]; everything else as vt_patch_embed_gemm, which is this function at H = W = S.
 * Replaces ViTPatchEmbeddings.forward(pixel_values, interpolate_pos_encoding=True) plus the CLS / position add of
 * ViTEmbeddings.forward (transformers/models/vit/modeling_vit.py). */
int vt_patch_embed_gemm_hw(const void* pixels, int32_t pix_dtype, const void* w, int64_t ldw, const float* bias,
                           const void* posb, void* out, float* stats_out, void* workspace, int32_t B, int32_t C,
                           int32_t H, int32_t W, int32_t P, int32_t D, void* stream);

/* Position table resample: pos [1 + g_in^2, D] (pos_dtype f32|bf16) -> out f32 [1 + gh*gw, D].  Row 0 (CLS) is copied;
 * rows >= 1 are F.interpolate(grid, size=(gh, gw), mode="bicubic", align_corners=False) of the g_in x g_in grid,
 * channel last, in fp32 (Keys cubic A = -0.75, clamped taps, horizontal pass first); gh = gw = g_in reproduces the
 * input exactly.  pos and out must not overlap.
 * Replaces ViTEmbeddings.interpolate_pos_encoding (transformers/models/vit/modeling_vit.py). */
int vt_pos_embed_resample(const void* pos, int32_t pos_dtype, float* out, int32_t D, int32_t g_in, int32_t gh,
                          int32_t gw, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* VITB200_RESOLUTION_H_ */
