#include "kernels.cuh"

#include <cmath>
#include <mutex>
#include <vector>

namespace mb {
namespace kernels {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

// ------------------------------------------------------------------------------------------------ LayerNorm
// One warp per row, the whole row lives in registers (two-pass mean / variance like torch's CPU kernel).
constexpr int LN_MAX_V4 = 8;  // w <= 1024

template <bool GATHER_EMBED>
__device__ __forceinline__ void ln_row(float4 (&v)[LN_MAX_V4], int nv, int w, const float* gamma, const float* beta,
                                       float eps, int lane, float* of, __nv_bfloat16* ob) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < LN_MAX_V4; ++j)
        if (j < nv) s += v[j].x + v[j].y + v[j].z + v[j].w;
    const float mean = warp_sum(s) / (float)w;
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < LN_MAX_V4; ++j)
        if (j < nv) {
            const float a = v[j].x - mean, b = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
            q += a * a + b * b + c * c + d * d;
        }
    const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)w + eps);
#pragma unroll
    for (int j = 0; j < LN_MAX_V4; ++j)
        if (j < nv) {
            const int i4 = lane + 32 * j;
            const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + i4);
            const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + i4);
            float4 y;
            y.x = (v[j].x - mean) * rstd * g.x + b.x;
            y.y = (v[j].y - mean) * rstd * g.y + b.y;
            y.z = (v[j].z - mean) * rstd * g.z + b.z;
            y.w = (v[j].w - mean) * rstd * g.w + b.w;
            if (of) reinterpret_cast<float4*>(of)[i4] = y;
            if (ob) reinterpret_cast<uint2*>(ob)[i4] = make_uint2(pack_bf16x2(y.x, y.y), pack_bf16x2(y.z, y.w));
        }
}

// Rows are visited LAST FIRST (block 0 takes the highest rows): the GEMM that produced x wrote its row bands in ascending
// order, so the rows it wrote last — the ones most likely still in the 126 MB L2 — are read first, and the bf16 rows this
// kernel writes last are the low ones the next GEMM (ascending again) starts with.
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, long long in_stride,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        float eps, int rows, int w, float* out_f32,
                                                        __nv_bfloat16* out_bf16) {
    int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    row = rows - 1 - row;
    const int nv = w / 128;
    const float4* src = reinterpret_cast<const float4*>(x + (long long)row * in_stride);
    float4 v[LN_MAX_V4];
#pragma unroll
    for (int j = 0; j < LN_MAX_V4; ++j)
        if (j < nv) v[j] = src[lane + 32 * j];
    ln_row<false>(v, nv, w, gamma, beta, eps, lane, out_f32 ? out_f32 + (long long)row * w : nullptr,
                  out_bf16 ? out_bf16 + (long long)row * w : nullptr);
}

static void check_ln_width(int w) {
    if (w % 128 != 0 || w > 128 * LN_MAX_V4) fail(B200_ERR_UNSUPPORTED, "width %d must be a multiple of 128 and <= 1024", w);
}

void layernorm(const float* x, long long in_stride, const float* gamma, const float* beta, float eps, int rows, int w,
               float* out_f32, __nv_bfloat16* out_bf16, cudaStream_t s) {
    if (rows <= 0) return;
    check_ln_width(w);
    layernorm_kernel<<<(rows + 7) / 8, 256, 0, s>>>(x, in_stride, gamma, beta, eps, rows, w, out_f32, out_bf16);
    MB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------ im2col
template <bool U8>
__global__ void __launch_bounds__(256) im2col_kernel(const void* __restrict__ img, int n, int S, int p, int kpad,
                                                     float3 scale, float3 shift, __nv_bfloat16* __restrict__ out) {
    // one thread = 8 consecutive k of one patch row
    const int g = S / p;
    const int groups = kpad / 8;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)n * g * g * groups;
    if (gid >= total) return;
    const int kg = (int)(gid % groups);
    const long long prow = gid / groups;
    const int px = (int)(prow % g);
    const int py = (int)((prow / g) % g);
    const long long b = prow / ((long long)g * g);
    const int K = 3 * p * p;
    float f[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int k = kg * 8 + e;
        float val = 0.f;
        if (k < K) {
            const int c = k / (p * p);
            const int rem = k - c * p * p;
            const int dy = rem / p, dx = rem - dy * p;
            const int y = py * p + dy, x = px * p + dx;
            if (U8) {
                const uint8_t u = reinterpret_cast<const uint8_t*>(img)[((b * S + y) * S + x) * 3 + c];
                const float sc = c == 0 ? scale.x : (c == 1 ? scale.y : scale.z);
                const float sh = c == 0 ? shift.x : (c == 1 ? shift.y : shift.z);
                // ToTensor then Normalize: (u/255 - mean)/std, evaluated as torchvision does (div, sub, div)
                val = ((float)u / 255.0f - sh) / sc;
            } else {
                val = reinterpret_cast<const float*>(img)[((b * 3 + c) * S + y) * S + x];
            }
        }
        f[e] = val;
    }
    reinterpret_cast<uint4*>(out)[gid] =
        make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
}

void im2col_u8(const uint8_t* img, int n, int S, int p, int kpad, const float* mean3, const float* std3,
               __nv_bfloat16* out, cudaStream_t s) {
    if (n <= 0) return;
    const int g = S / p;
    const long long total = (long long)n * g * g * (kpad / 8);
    const float3 sc = make_float3(std3[0], std3[1], std3[2]);
    const float3 sh = make_float3(mean3[0], mean3[1], mean3[2]);
    im2col_kernel<true><<<(unsigned)((total + 255) / 256), 256, 0, s>>>(img, n, S, p, kpad, sc, sh, out);
    MB_CUDA(cudaGetLastError());
}

void im2col_f32(const float* chw, int n, int S, int p, int kpad, __nv_bfloat16* out, cudaStream_t s) {
    if (n <= 0) return;
    const int g = S / p;
    const long long total = (long long)n * g * g * (kpad / 8);
    im2col_kernel<false><<<(unsigned)((total + 255) / 256), 256, 0, s>>>(chw, n, S, p, kpad, make_float3(1, 1, 1),
                                                                        make_float3(0, 0, 0), out);
    MB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------ embeddings
__global__ void vit_cls_kernel(float* x, const float* __restrict__ cls, const float* __restrict__ pos, int n,
                               int tokens_per_image, int w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * w) return;
    const int b = i / w, c = i - b * w;
    x[(long long)b * tokens_per_image * w + c] = cls[c] + pos[c];
}

void vit_cls_rows(float* x, const float* cls, const float* pos, int n, int tokens_per_image, int w, cudaStream_t s) {
    if (n <= 0) return;
    vit_cls_kernel<<<(n * w + 255) / 256, 256, 0, s>>>(x, cls, pos, n, tokens_per_image, w);
    MB_CUDA(cudaGetLastError());
}

__global__ void __launch_bounds__(256) clip_text_embed_kernel(const int32_t* __restrict__ ids, const float* __restrict__ tok,
                                                              const float* __restrict__ pos, int n, int S, int w, int vocab,
                                                              float* __restrict__ x, int32_t* __restrict__ eot) {
    // one warp per token row
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= (long long)n * S) return;
    const int s = (int)(row % S);
    int id = ids[row];
    id = min(max(id, 0), vocab - 1);
    const float4* t4 = reinterpret_cast<const float4*>(tok + (long long)id * w);
    const float4* p4 = reinterpret_cast<const float4*>(pos + (long long)s * w);
    float4* o4 = reinterpret_cast<float4*>(x + row * w);
    for (int i = lane; i < w / 4; i += 32) {
        const float4 a = __ldg(t4 + i), b = __ldg(p4 + i);
        o4[i] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    }
    if (s == 0 && lane == 0) {
        // torch.argmax: first occurrence of the maximum id
        const int32_t* r = ids + row;
        int best = 0, bv = r[0];
        for (int j = 1; j < S; ++j)
            if (r[j] > bv) {
                bv = r[j];
                best = j;
            }
        eot[row / S] = best;
    }
}

void clip_text_embed(const int32_t* ids, const float* tok, const float* pos, int n, int S, int w, int vocab, float* x,
                     int32_t* eot, cudaStream_t s) {
    if (n <= 0) return;
    const long long rows = (long long)n * S;
    clip_text_embed_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(ids, tok, pos, n, S, w, vocab, x, eot);
    MB_CUDA(cudaGetLastError());
}

// MPNET: no token-type row, and the position id of token s is 2 + s (1, the padding index, for pad tokens): HF's
// create_position_ids_from_input_ids on the right-padded rows the tokenizer produces
template <bool MPNET>
__global__ void __launch_bounds__(256) bert_embed_ln_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ mask,
                                                            const float* __restrict__ word, const float* __restrict__ pos,
                                                            const float* __restrict__ type0, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float eps, int n, int S, int w,
                                                            int vocab, float* __restrict__ x, __nv_bfloat16* __restrict__ h,
                                                            int32_t* __restrict__ kv_len) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= (long long)n * S) return;
    const int s = (int)(row % S);
    int id = ids[row];
    id = min(max(id, 0), vocab - 1);
    const int nv = w / 128;
    const float4* w4 = reinterpret_cast<const float4*>(word + (long long)id * w);
    const int p = MPNET ? ((mask == nullptr || mask[row] != 0) ? 2 + s : 1) : s;
    const float4* p4 = reinterpret_cast<const float4*>(pos + (long long)p * w);
    const float4* t4 = reinterpret_cast<const float4*>(type0);
    float4 v[LN_MAX_V4];
#pragma unroll
    for (int j = 0; j < LN_MAX_V4; ++j)
        if (j < nv) {
            const int i4 = lane + 32 * j;
            if constexpr (MPNET) {   // HF: inputs_embeds + position_embeddings
                const float4 a = __ldg(w4 + i4), b = __ldg(p4 + i4);
                v[j] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
            } else {
                const float4 a = __ldg(w4 + i4), b = __ldg(p4 + i4), c = __ldg(t4 + i4);
                // HF: inputs_embeds + token_type_embeddings, then + position_embeddings
                v[j] = make_float4((a.x + c.x) + b.x, (a.y + c.y) + b.y, (a.z + c.z) + b.z, (a.w + c.w) + b.w);
            }
        }
    ln_row<true>(v, nv, w, gamma, beta, eps, lane, x + row * w, h + row * w);
    if (s == 0 && lane == 0) {
        int cnt = S;
        if (mask) {
            cnt = 0;
            for (int j = 0; j < S; ++j) cnt += mask[row + j] != 0;
        }
        kv_len[row / S] = cnt;
    }
}

void bert_embed_ln(const int32_t* ids, const int32_t* mask, const float* word, const float* pos, const float* type0,
                   const float* gamma, const float* beta, float eps, int n, int S, int w, int vocab, float* x,
                   __nv_bfloat16* h, int32_t* kv_len, cudaStream_t s) {
    if (n <= 0) return;
    check_ln_width(w);
    const long long rows = (long long)n * S;
    bert_embed_ln_kernel<false><<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(ids, mask, word, pos, type0, gamma, beta, eps, n,
                                                                          S, w, vocab, x, h, kv_len);
    MB_CUDA(cudaGetLastError());
}

void mpnet_embed_ln(const int32_t* ids, const int32_t* mask, const float* word, const float* pos, const float* gamma,
                    const float* beta, float eps, int n, int S, int w, int vocab, float* x, __nv_bfloat16* h,
                    int32_t* kv_len, cudaStream_t s) {
    if (n <= 0) return;
    check_ln_width(w);
    const long long rows = (long long)n * S;
    bert_embed_ln_kernel<true><<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(ids, mask, word, pos, nullptr, gamma, beta, eps, n,
                                                                         S, w, vocab, x, h, kv_len);
    MB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------ heads
__device__ __forceinline__ float block_sum_256(float v, float* red) {
    v = warp_sum(v);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i];
    return t;
}

// CLIP head in three small kernels with enough parallelism to be latency-free:
//   (1) head_ln_kernel      one warp per image: gather the pooled token row, LayerNorm -> pooled fp32 [n, w]
//   (2) head_proj_kernel    grid (n/4, E/64): 4 images x 64 outputs per CTA, K split over 4 thread groups
//   (3) head_norm_kernel    one warp per image: L2 normalise (no epsilon, abstract_clip_model.py:83-85)
constexpr int HEAD_IMGS = 4;
constexpr int HEAD_COLS = 64;

__global__ void __launch_bounds__(256) head_ln_kernel(const float* __restrict__ x, int S, const int32_t* __restrict__ row_in_seq,
                                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                                      float eps, int n, int w, float* __restrict__ pooled) {
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (b >= n) return;
    const int r = row_in_seq ? row_in_seq[b] : 0;
    const float* src = x + ((long long)b * S + r) * w;
    float s = 0.f;
    for (int i = lane; i < w; i += 32) s += src[i];
    const float mean = warp_sum(s) / (float)w;
    float q = 0.f;
    for (int i = lane; i < w; i += 32) {
        const float d = src[i] - mean;
        q += d * d;
    }
    const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)w + eps);
    for (int i = lane; i < w; i += 32) pooled[(long long)b * w + i] = (src[i] - mean) * rstd * gamma[i] + beta[i];
}

__global__ void __launch_bounds__(256) head_proj_kernel(const float* __restrict__ pooled, const float* __restrict__ proj, int n,
                                                        int w, int E, float* __restrict__ out) {
    __shared__ float part[4][HEAD_IMGS][HEAD_COLS];
    extern __shared__ float s_pool[];   // [HEAD_IMGS][w]
    const int b0 = blockIdx.x * HEAD_IMGS;
    const int e = blockIdx.y * HEAD_COLS + (threadIdx.x & (HEAD_COLS - 1));
    const int slice = threadIdx.x >> 6;   // 4 K-slices
    for (int i = threadIdx.x; i < HEAD_IMGS * w; i += 256) {
        const int k = i / w, c = i - k * w;
        s_pool[i] = b0 + k < n ? pooled[(long long)(b0 + k) * w + c] : 0.f;
    }
    __syncthreads();
    float acc[HEAD_IMGS];
#pragma unroll
    for (int k = 0; k < HEAD_IMGS; ++k) acc[k] = 0.f;
    const int i0 = slice * (w / 4), i1 = i0 + w / 4;
    if (e < E) {
#pragma unroll 8
        for (int i = i0; i < i1; ++i) {
            const float pj = __ldg(proj + (long long)i * E + e);
#pragma unroll
            for (int k = 0; k < HEAD_IMGS; ++k) acc[k] = fmaf(s_pool[k * w + i], pj, acc[k]);
        }
    }
#pragma unroll
    for (int k = 0; k < HEAD_IMGS; ++k) part[slice][k][threadIdx.x & (HEAD_COLS - 1)] = acc[k];
    __syncthreads();
    if (slice == 0 && e < E) {
#pragma unroll
        for (int k = 0; k < HEAD_IMGS; ++k)
            if (b0 + k < n) {
                const int c = threadIdx.x & (HEAD_COLS - 1);
                // fixed order: the result does not depend on scheduling
                out[(long long)(b0 + k) * E + e] = ((part[0][k][c] + part[1][k][c]) + part[2][k][c]) + part[3][k][c];
            }
    }
}

__global__ void __launch_bounds__(256) head_norm_kernel(float* __restrict__ out, int n, int E) {
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (b >= n) return;
    float* row = out + (long long)b * E;
    float ss = 0.f;
    for (int i = lane; i < E; i += 32) ss += row[i] * row[i];
    const float nrm = sqrtf(warp_sum(ss));
    for (int i = lane; i < E; i += 32) row[i] = row[i] / nrm;
}

void clip_head(const float* x, int S, const int32_t* row_in_seq, const float* gamma, const float* beta, float eps,
               const float* proj, int n, int w, int E, int normalize, float* out, float* pooled_ws, cudaStream_t s) {
    if (n <= 0) return;
    if (w % 4 != 0 || (size_t)HEAD_IMGS * w * sizeof(float) > 40 * 1024)
        fail(B200_ERR_UNSUPPORTED, "clip_head: width %d unsupported", w);
    head_ln_kernel<<<(n + 7) / 8, 256, 0, s>>>(x, S, row_in_seq, gamma, beta, eps, n, w, pooled_ws);
    MB_CUDA(cudaGetLastError());
    const dim3 grid((n + HEAD_IMGS - 1) / HEAD_IMGS, (E + HEAD_COLS - 1) / HEAD_COLS);
    head_proj_kernel<<<grid, 256, (size_t)HEAD_IMGS * w * sizeof(float), s>>>(pooled_ws, proj, n, w, E, out);
    MB_CUDA(cudaGetLastError());
    if (normalize) {
        head_norm_kernel<<<(n + 7) / 8, 256, 0, s>>>(out, n, E);
        MB_CUDA(cudaGetLastError());
    }
}

__global__ void __launch_bounds__(256) bert_head_kernel(const float* __restrict__ x, const int32_t* __restrict__ kv_len, int S,
                                                        int w, int pool, int normalize, float* __restrict__ out) {
    __shared__ float red[8];
    const int b = blockIdx.x;
    const int len = min(max(kv_len[b], 0), S);
    const float* src = x + (long long)b * S * w;
    float vals[4];  // w <= 1024
    float ss = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int i = threadIdx.x + 256 * j;
        float v = 0.f;
        if (i < w) {
            if (pool == 1) {
                v = src[i];
            } else {
                float acc = 0.f;
                for (int t = 0; t < len; ++t) acc += src[(long long)t * w + i];
                v = acc / (float)len;  // len == 0 -> NaN, as sum / 0 does in the reference
            }
            ss += v * v;
        }
        vals[j] = v;
    }
    const float nrm = fmaxf(sqrtf(block_sum_256(ss, red)), 1e-12f);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int i = threadIdx.x + 256 * j;
        if (i < w) out[(long long)b * w + i] = normalize ? vals[j] / nrm : vals[j];
    }
}

void bert_head(const float* x, const int32_t* kv_len, int n, int S, int w, int pool, int normalize, float* out,
               cudaStream_t s) {
    if (n <= 0) return;
    if (w > 1024) fail(B200_ERR_UNSUPPORTED, "bert_head: width %d > 1024", w);
    bert_head_kernel<<<n, 256, 0, s>>>(x, kv_len, S, w, pool, normalize, out);
    MB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------ conversions
__global__ void f32_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = __float2bfloat16_rn(src[i]);
}
void f32_to_bf16(const float* src, __nv_bfloat16* dst, long long n, cudaStream_t s) {
    if (n <= 0) return;
    f32_to_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, dst, n);
    MB_CUDA(cudaGetLastError());
}

__global__ void pad_rows_kernel(const float* __restrict__ src, int rows, int k, int kpad, __nv_bfloat16* __restrict__ dst) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)rows * kpad) return;
    const int r = (int)(i / kpad), c = (int)(i % kpad);
    dst[i] = __float2bfloat16_rn(c < k ? src[(long long)r * k + c] : 0.f);
}
void pad_rows_to_bf16(const float* src, int rows, int k, int kpad, __nv_bfloat16* dst, cudaStream_t s) {
    const long long n = (long long)rows * kpad;
    pad_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, rows, k, kpad, dst);
    MB_CUDA(cudaGetLastError());
}

// conv1.weight [w, 3, p, p] -> the gather GEMM's K order: k' = dy * (64 * kbpd) + dx * 3 + c, zero in the padding slots
__global__ void patch_weight_rows_kernel(const float* __restrict__ src, int rows, int p, int kbpd,
                                         __nv_bfloat16* __restrict__ dst) {
    const int kprime = p * kbpd * 64;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)rows * kprime) return;
    const int r = (int)(i / kprime), k = (int)(i - (long long)r * kprime);
    const int dy = k / (64 * kbpd), q = k - dy * 64 * kbpd;
    float v = 0.f;
    if (q < 3 * p) {
        const int dx = q / 3, c = q - 3 * dx;
        v = src[(long long)r * 3 * p * p + (long long)c * p * p + dy * p + dx];
    }
    dst[i] = __float2bfloat16_rn(v);
}
void patch_weight_rows(const float* src, int rows, int p, int kbpd, __nv_bfloat16* dst, cudaStream_t s) {
    const long long n = (long long)rows * p * kbpd * 64;
    patch_weight_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, rows, p, kbpd, dst);
    MB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------ resize
// Pillow's ImagingResample for 8-bit images, restated: per-output-pixel coefficient windows computed in double on
// the host exactly as precompute_coeffs()/normalize_coeffs_8bpc() do (bicubic a = -0.5, support widened by the
// down-scale factor, coefficients rounded to 22-bit fixed point), horizontal pass into an 8-bit intermediate, then
// the vertical pass; each pass accumulates in int32 starting from 1 << 21 and clips (x >> 22) to [0, 255].
constexpr int PRECISION_BITS = 32 - 8 - 2;

struct ResampleTable {
    int ksize = 0;
    std::vector<int> bounds;  // [out][2] = (xmin, xcount)
    std::vector<int> coeffs;  // [out][ksize]
};

static double bicubic_filter(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}

static ResampleTable precompute(int in_size, int out_size) {
    ResampleTable t;
    const double scale = (double)in_size / (double)out_size;
    double filterscale = scale;
    if (filterscale < 1.0) filterscale = 1.0;
    const double support = 2.0 * filterscale;
    t.ksize = (int)ceil(support) * 2 + 1;
    t.bounds.assign((size_t)out_size * 2, 0);
    t.coeffs.assign((size_t)out_size * t.ksize, 0);
    std::vector<double> k(t.ksize);
    for (int xx = 0; xx < out_size; ++xx) {
        const double center = (xx + 0.5) * scale;
        double ww = 0.0;
        const double ss = 1.0 / filterscale;
        int xmin = (int)(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = (int)(center + support + 0.5);
        if (xmax > in_size) xmax = in_size;
        xmax -= xmin;
        for (int x = 0; x < xmax; ++x) {
            const double w = bicubic_filter((x + xmin - center + 0.5) * ss);
            k[x] = w;
            ww += w;
        }
        for (int x = 0; x < xmax; ++x)
            if (ww != 0.0) k[x] /= ww;
        for (int x = 0; x < t.ksize; ++x) {
            const double v = x < xmax ? k[x] : 0.0;
            t.coeffs[(size_t)xx * t.ksize + x] =
                v < 0 ? (int)(-0.5 + v * (1 << PRECISION_BITS)) : (int)(0.5 + v * (1 << PRECISION_BITS));
        }
        t.bounds[xx * 2] = xmin;
        t.bounds[xx * 2 + 1] = xmax;
    }
    return t;
}

__device__ __forceinline__ uint8_t clip8(int v) {
    v >>= PRECISION_BITS;
    return (uint8_t)min(max(v, 0), 255);
}

// horizontal: src [n, h, w, 3] -> tmp [n, h, S, 3] for output columns x_off .. x_off + S - 1 of the resized image
__global__ void resample_h_kernel(const uint8_t* __restrict__ src, int n, int h, int w, int S, int x_off,
                                  const int* __restrict__ bounds, const int* __restrict__ coeffs, int ksize,
                                  uint8_t* __restrict__ tmp) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n * h * S) return;
    const int xo = (int)(i % S);
    const long long rowi = i / S;  // (image, y)
    const int xx = xo + x_off;
    const int xmin = bounds[xx * 2], cnt = bounds[xx * 2 + 1];
    const int* k = coeffs + (long long)xx * ksize;
    const uint8_t* line = src + rowi * w * 3;
    int s0 = 1 << (PRECISION_BITS - 1), s1 = s0, s2 = s0;
    for (int x = 0; x < cnt; ++x) {
        const int c = k[x];
        const uint8_t* px = line + (xmin + x) * 3;
        s0 += px[0] * c;
        s1 += px[1] * c;
        s2 += px[2] * c;
    }
    uint8_t* o = tmp + i * 3;
    o[0] = clip8(s0);
    o[1] = clip8(s1);
    o[2] = clip8(s2);
}

// vertical: tmp [n, h, S, 3] -> dst [n, S, S, 3] for output rows y_off .. y_off + S - 1
__global__ void resample_v_kernel(const uint8_t* __restrict__ tmp, int n, int h, int S, int y_off,
                                  const int* __restrict__ bounds, const int* __restrict__ coeffs, int ksize,
                                  uint8_t* __restrict__ dst) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n * S * S) return;
    const int xo = (int)(i % S);
    const int yo = (int)((i / S) % S);
    const long long b = i / ((long long)S * S);
    const int yy = yo + y_off;
    const int ymin = bounds[yy * 2], cnt = bounds[yy * 2 + 1];
    const int* k = coeffs + (long long)yy * ksize;
    int s0 = 1 << (PRECISION_BITS - 1), s1 = s0, s2 = s0;
    for (int y = 0; y < cnt; ++y) {
        const int c = k[y];
        const uint8_t* px = tmp + ((b * h + ymin + y) * S + xo) * 3;
        s0 += px[0] * c;
        s1 += px[1] * c;
        s2 += px[2] * c;
    }
    uint8_t* o = dst + i * 3;
    o[0] = clip8(s0);
    o[1] = clip8(s1);
    o[2] = clip8(s2);
}

static int py_round_half_even(double v) { return (int)nearbyint(v); }

void resize_crop_u8(const uint8_t* src, int n, int h, int w, int S, uint8_t* dst, cudaStream_t s) {
    if (n <= 0) return;
    // torchvision Resize(S): shortest side -> S, the other int(S * long / short); CenterCrop(S)
    int new_w, new_h;
    if (w <= h) {
        new_w = S;
        new_h = (int)((double)((long long)S * h) / (double)w);  // int(S * long / short): Python true division
    } else {
        new_h = S;
        new_w = (int)((double)((long long)S * w) / (double)h);
    }
    const int left = py_round_half_even((new_w - S) / 2.0);
    const int top = py_round_half_even((new_h - S) / 2.0);
    const ResampleTable th = precompute(w, new_w);
    const ResampleTable tv = precompute(h, new_h);
    int *d_hb = nullptr, *d_hc = nullptr, *d_vb = nullptr, *d_vc = nullptr;
    uint8_t* tmp = nullptr;
    auto up = [&](const std::vector<int>& v, int** d) {
        MB_CUDA(cudaMallocAsync((void**)d, v.size() * sizeof(int), s));
        MB_CUDA(cudaMemcpyAsync(*d, v.data(), v.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    };
    up(th.bounds, &d_hb);
    up(th.coeffs, &d_hc);
    up(tv.bounds, &d_vb);
    up(tv.coeffs, &d_vc);
    MB_CUDA(cudaMallocAsync((void**)&tmp, (size_t)n * h * S * 3, s));
    // the pageable host vectors above must outlive the async copies: synchronise before they go out of scope
    const long long nh = (long long)n * h * S;
    resample_h_kernel<<<(unsigned)((nh + 255) / 256), 256, 0, s>>>(src, n, h, w, S, left, d_hb, d_hc, th.ksize, tmp);
    MB_CUDA(cudaGetLastError());
    const long long nv = (long long)n * S * S;
    resample_v_kernel<<<(unsigned)((nv + 255) / 256), 256, 0, s>>>(tmp, n, h, S, top, d_vb, d_vc, tv.ksize, dst);
    MB_CUDA(cudaGetLastError());
    MB_CUDA(cudaFreeAsync(d_hb, s));
    MB_CUDA(cudaFreeAsync(d_hc, s));
    MB_CUDA(cudaFreeAsync(d_vb, s));
    MB_CUDA(cudaFreeAsync(d_vc, s));
    MB_CUDA(cudaFreeAsync(tmp, s));
    MB_CUDA(cudaStreamSynchronize(s));
}

}  // namespace kernels
}  // namespace mb
