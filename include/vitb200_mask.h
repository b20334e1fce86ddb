/*
 * vitb200_mask.h — entry points of libvitb200.so for masked inputs (HF ViTModel's bool_masked_pos) and the masked
 * image modeling head of ViTForMaskedImageModeling (SimMIM): masked patches take the mask token instead of their
 * projection, the decoder's 1x1 convolution output is pixel-shuffled back into an image, and the L1 loss over the
 * masked pixels is reduced on the device.
 *
 * Same conventions as vitb200.h (device pointers, dtype codes, void* stream, 0 / negative vt_status / positive
 * cudaError_t, no synchronisation, no device allocation, safe inside CUDA-graph capture: the mask is read on the
 * device), and exported from the same library.  They are declared here rather than in vitb200.h so that the core
 * header's entry-point set stays fixed.  mask is always a device bool (one byte, 0 / 1) array [B, gh * gw] in patch
 * order; patch p of an image is token 1 + p.
 */
#ifndef VITB200_MASK_H_
#define VITB200_MASK_H_

#include "vitb200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Masked patch gather: pixels [B,C,H,W] (pix_dtype f32|bf16) or [B,H,W,C] (VT_U8), grid gh x gw = (H / P) x (W / P)
 * rounded down, N = 1 + gh * gw rows per image, unpadded.  Writes
 *   patches bf16 [B * N, ldw]: row b * N + 1 + p = pixels of patch p in the order of vt_patch_embed_gemm_hw, zero when
 *                              mask[b, p] (its pixels are not read); the CLS rows and the columns K .. ldw zero;
 *   table   bf16 [B * N, D]:   row b * N + t = posm[t] when t >= 1 and mask[b, t - 1], else pos[t].
 * pos bf16 [N, D] is the table of vt_patch_embed_gemm_hw (row 0 = cls + pos[0] - bias); posm bf16 [N, D] is
 * mask_token + pos - bias (row 0 is not read).  vt_gemm_bf16_ln(patches, ldw, w, ldw, out, D, bias, table, D, B * N,
 * D, ldw, ...) then gives the embeddings (and row statistics), and with an all-false mask exactly what
 * vt_patch_embed_gemm_hw gives.  K = C * P * P <= ldw, ldw % 8 == 0, D % 8 == 0, B <= 65535, B * N < 2^31; pixels,
 * patches, table, pos and posm 16-byte aligned.  Replaces ViTPatchEmbeddings.forward plus the mask-token blend and
 * the CLS / position add of ViTEmbeddings.forward(pixel_values, bool_masked_pos) (transformers/models/vit/
 * modeling_vit.py). */
int vt_patch_embed_masked_gather(const void* pixels, int32_t pix_dtype, const void* mask, const void* pos,
                                 const void* posm, void* patches, int64_t ldw, void* table, int32_t B, int32_t C,
                                 int32_t H, int32_t W, int32_t P, int32_t D, void* stream);

/* vt_embed_finalize with a mask: x [B, N, D] (dtype f32|bf16) holds the patch projections in rows 1 .. N - 1;
 * x[b, 0] = cls + pos[0], x[b, t] = (mask[b, t - 1] ? mask_token : x[b, t]) + pos[t], in fp32, rounded once.
 * pos [N, D], cls [D], mask_token [D] in the same dtype. */
int vt_embed_finalize_masked(void* x, const void* pos, const void* cls, const void* mask_token, const void* mask,
                             int32_t B, int32_t N, int32_t D, int32_t dtype, void* stream);

/* Masked image modeling reconstruction: dec [B, 1 + gh * gw, s * s * C] (dtype f32|bf16) is the decoder's 1x1
 * convolution over the final hidden states, row 0 of each image (CLS) is skipped; rec [B, C, gh * s, gw * s] (same
 * dtype) = PixelShuffle(s) of it: rec[b, c, y * s + i, x * s + j] = dec[b, 1 + y * gw + x, (c * s + i) * s + j].
 * With loss != NULL (needs mask, pixels and partial, and H = gh * s, W = gw * s pixels) it also writes
 *   *loss = sum over masked patches of |pixel - rec| / (masked patches * s * s + 1e-5) / C
 * as a 0-dim fp32 value: HF's masked L1 loss.  pixels [B, C, H, W] (pix_dtype f32|bf16) or [B, H, W, C] (VT_U8,
 * normalised on the fly as (u * rescale - norm[c]) / norm[C + c], norm fp32 [2C] = mean, std).  partial fp32
 * [B * gh * gw] is scratch; the sums run in a fixed order, so the loss is the same bit for bit on every call.
 * Replaces ViTForMaskedImageModeling.forward's decoder PixelShuffle and loss (transformers/models/vit/
 * modeling_vit.py). */
int vt_mim_reconstruct(const void* dec, void* rec, int32_t dtype, int32_t B, int32_t C, int32_t gh, int32_t gw,
                       int32_t s, const void* pixels, int32_t pix_dtype, const float* norm, float rescale,
                       const void* mask, float* partial, float* loss, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* VITB200_MASK_H_ */
