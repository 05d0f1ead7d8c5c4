// Memory-bound helper kernels of the encoders (LayerNorm, embeddings, im2col + image normalise, pooling +
// projection + L2 normalise, dtype conversion).  All are coalesced / vectorised; none is GEMM-shaped.
#pragma once
#include "common.cuh"

namespace mb {
namespace kernels {

// y = LayerNorm(x) * gamma + beta over rows of width w (w % 128 == 0, w <= 1024).  Row r is read at
// x + r * in_stride (floats).  Writes fp32 (out_f32, may alias x) and/or bf16 (out_bf16), both compact [rows, w].
void layernorm(const float* x, long long in_stride, const float* gamma, const float* beta, float eps, int rows, int w,
               float* out_f32, __nv_bfloat16* out_bf16, cudaStream_t s);

// uint8 HWC images [n, S, S, 3] -> normalised bf16 patch matrix [n * g * g, kpad], k = c*p*p + dy*p + dx
// ((u8/255 - mean[c]) / std[c]; zero for k >= 3*p*p).  This is the CLIP ToTensor + Normalize fused into im2col.
void im2col_u8(const uint8_t* img, int n, int S, int p, int kpad, const float* mean3, const float* std3,
               __nv_bfloat16* out, cudaStream_t s);
// Already-normalised fp32 CHW [n, 3, S, S] -> bf16 patch matrix.
void im2col_f32(const float* chw, int n, int S, int p, int kpad, __nv_bfloat16* out, cudaStream_t s);

// x[b*(G+1), :] = class_embedding + positional_embedding[0]
void vit_cls_rows(float* x, const float* cls, const float* pos, int n, int tokens_per_image, int w, cudaStream_t s);

// CLIP text: x[b, s, :] = token_embedding[ids[b, s]] + positional_embedding[s]; also eot[b] = arg-max_s ids[b, s]
void clip_text_embed(const int32_t* ids, const float* tok, const float* pos, int n, int S, int w, int vocab, float* x,
                     int32_t* eot, cudaStream_t s);

// BERT: x = LN(word[ids] + position[s] + token_type[0]); fp32 + bf16 copies.  Also kv_len[b] = sum(mask[b, :])
// (mask may be NULL = all ones).
void bert_embed_ln(const int32_t* ids, const int32_t* mask, const float* word, const float* pos, const float* type0,
                   const float* gamma, const float* beta, float eps, int n, int S, int w, int vocab, float* x,
                   __nv_bfloat16* h, int32_t* kv_len, cudaStream_t s);
// MPNet: x = LN(word[ids] + position[p]) with p = 2 + s for tokens (mask 1 or NULL) and p = 1 for pads; no token type.
// kv_len as bert_embed_ln.  position: [>= S + 2, w].
void mpnet_embed_ln(const int32_t* ids, const int32_t* mask, const float* word, const float* pos, const float* gamma,
                    const float* beta, float eps, int n, int S, int w, int vocab, float* x, __nv_bfloat16* h,
                    int32_t* kv_len, cudaStream_t s);

// CLIP head: for image b take token row (b * S + row_in_seq[b]) (row_in_seq NULL -> 0), LayerNorm it, multiply by
// proj [w, E] (fp32), optionally divide by the L2 norm (no epsilon: abstract_clip_model.py:83-85).
// pooled_ws: fp32 workspace [n, w].
void clip_head(const float* x, int S, const int32_t* row_in_seq, const float* gamma, const float* beta, float eps,
               const float* proj, int n, int w, int E, int normalize, float* out, float* pooled_ws, cudaStream_t s);

// BERT head: masked mean over the first kv_len[b] tokens (pool == 0) or the [CLS] row (pool == 1), then
// x / max(|x|, 1e-12) if normalize (F.normalize, hugging_face_model.py:194-195).
void bert_head(const float* x, const int32_t* kv_len, int n, int S, int w, int pool, int normalize, float* out,
               cudaStream_t s);

void f32_to_bf16(const float* src, __nv_bfloat16* dst, long long n, cudaStream_t s);
// conv1.weight [w, 3*p*p] -> bf16 [w, kpad] zero padded
void pad_rows_to_bf16(const float* src, int rows, int k, int kpad, __nv_bfloat16* dst, cudaStream_t s);

// conv1.weight [w, 3, p, p] (fp32) -> bf16 [w, p * kbpd * 64] in the gather GEMM's K order (gemm.cuh: PatchGather):
// k' = dy * (64 * kbpd) + dx * 3 + c; the slots past 3 * p of every pixel row are zero.
void patch_weight_rows(const float* src, int rows, int p, int kbpd, __nv_bfloat16* dst, cudaStream_t s);

// PIL-compatible antialiased bicubic resize (shortest side -> S) + centre crop, uint8 HWC in/out.
void resize_crop_u8(const uint8_t* src, int n, int h, int w, int S, uint8_t* dst, cudaStream_t s);

}  // namespace kernels
}  // namespace mb
