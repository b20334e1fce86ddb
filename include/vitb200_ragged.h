/*
 * vitb200_ragged.h — entry points of libvitb200.so that run images of different resolutions in ONE batch: the
 * images' tokens are packed into one [M, D] activation (M = sum of 1 + (H_i / P) * (W_i / P), no padding between
 * images), so every dense layer of the encoder is one launch over all of them.  Only the patch gather, the
 * position table and the attention depend on the image.
 *
 * Same conventions as vitb200.h (device pointers, dtype codes, void* stream, 0 / negative vt_status / positive
 * cudaError_t, no synchronisation, no device allocation), and exported from the same library.  They are declared here
 * rather than in vitb200.h so that the core header's entry-point set stays fixed.  HF ViTModel has no ragged batch;
 * the per-image result it stands for is ViTModel(pixel_values=image[None], interpolate_pos_encoding=True).
 */
#ifndef VITB200_RAGGED_H_
#define VITB200_RAGGED_H_

#include "vitb200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* One image of a ragged batch (40 bytes, the array lives in device memory). */
typedef struct vt_ragged_image {
  const void* pixels; /* [C, height, width] (f32 | bf16) or [height, width, C] (VT_U8), contiguous */
  const void* pos;    /* bf16 [tokens, D] position table of its grid, row 0 = cls + pos[0] - bias */
  int64_t row0;       /* first row of the image in the packed output */
  int32_t height;
  int32_t width;
  int32_t tokens;     /* 1 + (height / P) * (width / P) */
  int32_t reserved;   /* 0 */
} vt_ragged_image;

/* Ragged patch gather, one launch for the whole list: images [n_images] (device), sorted by row0, each image's rows
 * [row0, row0 + tokens) consecutive and together covering [0, M).  Writes
 *   patches bf16 [M, ldw]: row row0 + 1 + p = pixels of patch p in the order of vt_patch_embed_gemm_hw ((c, i, j) for
 *                          f32 / bf16 NCHW, (i, j, c) for uint8 NHWC); row row0 (CLS) and the columns K .. ldw zero;
 *                          the last height % P rows and width % P columns of an image belong to no patch;
 *   table   bf16 [M, D]:   row row0 + t = pos[t] of the image.
 * vt_gemm_bf16_ln(patches, ldw, w, ldw, out, D, bias, table, D, M, D, ldw, ...) then gives every image's embeddings
 * (and row statistics) exactly as vt_patch_embed_gemm_hw gives them for that image alone.  K = C * P * P <= ldw,
 * ldw % 8 == 0, D % 8 == 0, 0 < M < 2^31; patches and table 16-byte aligned.  Pixel rows whose image or width is not
 * 16-byte / 8-element aligned take the scalar loads.  Replaces, per image, ViTPatchEmbeddings.forward plus the CLS /
 * position add of ViTEmbeddings.forward with interpolate_pos_encoding=True (transformers/models/vit/modeling_vit.py). */
int vt_patch_embed_ragged_gather(const vt_ragged_image* images, int32_t n_images, int32_t pix_dtype, int32_t C,
                                 int32_t P, void* patches, int64_t ldw, void* table, int32_t D, int64_t M,
                                 void* stream);

/* Row gather: out[i, :cols] = x[idx[i], :cols] for i < rows (dtype f32 | bf16, idx int64 in device memory, row strides
 * in elements).  Collects the CLS rows of a ragged batch for the pooled output and the heads. */
int vt_gather_rows(const void* x, int64_t ldx, const int64_t* idx, void* out, int64_t ldo, int32_t rows, int32_t cols,
                   int32_t dtype, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* VITB200_RAGGED_H_ */
