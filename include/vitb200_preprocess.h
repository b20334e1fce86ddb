/*
 * vitb200_preprocess.h — entry points of libvitb200.so for the first step of HF's ViT image processor: the resize of
 * raw uint8 HWC images of any size to the model's size, byte for byte what PIL's Image.resize gives for BILINEAR and
 * BICUBIC (transformers ViTImageProcessorPil.resize; libImaging/Resample.c).  Rescale and normalisation are folded into
 * the patch embedding of the uint8 path (VT_U8 pixels), so resize + forward is the whole processor.
 *
 * Same conventions as vitb200.h (device pointers, void* stream, 0 / negative vt_status / positive cudaError_t, no
 * synchronisation, no device allocation, safe inside CUDA-graph capture: the tables and descriptors are read on the
 * device), and exported from the same library.  They are declared here rather than in vitb200.h so that the core
 * header's entry-point set stays fixed.
 *
 * Coefficient tables.  One table per axis (in -> out samples), built on the host (vit/kernels/resize.py): int32
 * [out][2 + k], entry o = start, count, then k weights w[0..k) in units of 2^-22, the first count of them used.
 * Output sample o reads input samples start + j for j < count only.  The caller guarantees 0 <= start,
 * 1 <= count <= k, start + count <= in, and start and start + count nondecreasing in o (true of PIL's tables); the
 * kernels index nothing else.  Each pass computes, per channel, clamp((2^21 + sum_j in[start + j] * w[j]) >> 22, 0, 255)
 * in exact int32 arithmetic: first along the width into a uint8 intermediate, then along the height from it (PIL's
 * order and rounding).  An image more than 100 times taller than wide whose height shrinks (H > 100 W, out_h < H) is
 * resized height first, as PIL 12's Image.resize does.  Channels (C <= 4) are resampled independently: PIL's L, RGB
 * and RGBX, not its alpha-premultiplied RGBA.
 */
#ifndef VITB200_PREPROCESS_H_
#define VITB200_PREPROCESS_H_

#include "vitb200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* One image of a resize list (40 bytes, the array lives in device memory). */
typedef struct vt_resize_image {
  const void* pixels; /* uint8 [height, width, C], contiguous */
  int64_t htab;       /* offset, in int32 elements of tables, of the width table [out_w][2 + hk] (width -> out_w) */
  int64_t vtab;       /* offset of the height table [out_h][2 + vk] (height -> out_h) */
  int32_t height;
  int32_t width;
  int32_t hk;         /* weights per entry of the width table */
  int32_t vk;         /* weights per entry of the height table */
} vt_resize_image;

/* Batch resize: src uint8 [B] images of [H, W, C] (each contiguous, batch_stride bytes apart, batch_stride >=
 * H * W * C) -> out uint8 [B, out_h, out_w, C] contiguous, with the width table htab [out_w][2 + hk] (W -> out_w) and
 * the height table vtab [out_h][2 + vk] (H -> out_h).  1 <= C <= 4, every size positive.  One launch (kernel
 * vt_resize_u8_kernel).  Replaces PIL.Image.resize(img, (out_w, out_h), BILINEAR | BICUBIC) per image. */
int vt_resize_u8(const void* src, int32_t B, int32_t H, int32_t W, int32_t C, int64_t batch_stride,
                 const int32_t* htab, int32_t hk, const int32_t* vtab, int32_t vk, void* out, int32_t out_h,
                 int32_t out_w, void* stream);

/* List resize: images [n_images] (device) of different sizes, each with its own tables inside tables (device int32)
 * -> out uint8 [n_images, out_h, out_w, C] contiguous, image i at out + i * out_h * out_w * C.  1 <= C <= 4. */
int vt_resize_u8_list(const vt_resize_image* images, int32_t n_images, int32_t C, const int32_t* tables, void* out,
                      int32_t out_h, int32_t out_w, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* VITB200_PREPROCESS_H_ */
