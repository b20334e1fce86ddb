/*
 * vitb200_attn.h — entry point of libvitb200.so for HF ViTModel's output_attentions: the attention probabilities
 * softmax(scale * Q K^T) of every head, written as a dense [B, H, N, N] tensor next to the fused attention of
 * vt_flash_attn, which never materialises them.
 *
 * Same conventions as vitb200.h (device pointers, void* stream, 0 / negative vt_status / positive cudaError_t, no
 * synchronisation, no device allocation, safe inside CUDA-graph capture), and exported from the same library.  It is
 * declared here rather than in vitb200.h so that the core header's entry-point set stays fixed.
 */
#ifndef VITB200_ATTN_H_
#define VITB200_ATTN_H_

#include "vitb200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Attention probabilities of the fused-QKV activation: q and k are bf16 views of its Q and K thirds, laid out as for
 * vt_flash_attn (head h at columns h * dh .. h * dh + dh - 1, qk_row_stride elements between tokens,
 * qk_batch_stride between images).  Writes
 *   probs bf16 [B, H, N, N], dense:  probs[b, h, i, j] = exp(s_ij - max_j s_ij) / sum_j exp(s_ij - max_j s_ij),
 *   s_ij = scale * q[b, i, h] . k[b, j, h] in fp32, each element rounded to bf16 once.
 * dh 64 or 80, any N >= 1, any B * H; scale > 0.  q, k 16-byte aligned, strides multiples of 8, probs 2-byte aligned;
 * no element outside probs[0 .. B * H * N * N) is written.  Anything else returns VT_ERR_UNSUPPORTED (shapes) or
 * VT_ERR_ALIGN.  Replaces the attention_probs that HF ViTSelfAttention returns with output_attentions=True
 * (transformers/models/vit/modeling_vit.py, eager attention). */
int vt_attn_probs(const void* q, const void* k, void* probs, int32_t B, int32_t H, int32_t N, int32_t dh,
                  int64_t qk_row_stride, int64_t qk_batch_stride, float scale, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* VITB200_ATTN_H_ */
