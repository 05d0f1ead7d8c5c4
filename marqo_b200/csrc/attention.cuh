// Multi-head attention over packed QKV (head_dim 64), flash-style online softmax in fp32.
//   129 <= S <= 257 without a bias: one-shot tcgen05 kernel (attention_os.cu) — all keys in one MMA.
//   every other input: tcgen05 / TMEM block kernel (attention_tc.cu) — 128 x 128 tiles, TMA-fed, thread-per-row
//             softmax; S < 128 packs several sequences into one tile under a block-diagonal mask.
#pragma once
#include "common.cuh"

namespace mb {
namespace attention {

enum Mask { MASK_NONE = 0, MASK_CAUSAL = 1, MASK_KEYLEN = 2 };

// Relative-position bias (MPNet): score(i, j) += rel_bias[bucket(j - i)][h], bucket = transformers'
// MPNetEncoder.relative_position_bucket with 32 buckets and max_distance 128.  Every |d| >= REL_D falls in the last
// bucket of its sign, so the kernels read the bias of a distance from a per-head row over d in [-REL_D, REL_D].
constexpr int REL_BUCKETS = 32;
constexpr int REL_D = 91;
constexpr int REL_T = 2 * REL_D + 1;   // entries per head of the folded table
// bucket of the distance d = key - query (host; fp32 log, as torch evaluates it)
int relative_position_bucket(int d);
// rel_bias fp32 [REL_BUCKETS, H] (host, the checkpoint's encoder.relative_attention_bias.weight) -> bias_log2 fp32
// [H, REL_T] (host): bias_log2[h][d + REL_D] = rel_bias[bucket(d)][h] * log2(e).  The bucket of every distance up to
// max_dist is checked to equal the bucket of the clamped distance.
void fold_relative_bias(const float* rel_bias, int H, int max_dist, float* bias_log2);

// qkv: bf16 [B*S, 3*W] rows = tokens, columns = [q | k | v], head h occupies columns h*64..h*64+63 of each part.
// out: bf16 [B*S, W].  kv_len: int32 [B] valid key count per sequence (MASK_KEYLEN only).
// bias_log2: device fp32 [H, REL_T] from fold_relative_bias, or nullptr for no bias (MASK_CAUSAL takes none).
// Returns the number of kernels launched.
int launch(const __nv_bfloat16* qkv, __nv_bfloat16* out, int B, int S, int W, int H, int mask, const int32_t* kv_len,
           const float* bias_log2, cudaStream_t stream);

// tcgen05 / TMEM implementation (attention_tc.cu)
int launch_tc(const __nv_bfloat16* qkv, __nv_bfloat16* out, int B, int S, int W, int H, int mask, const int32_t* kv_len,
              const float* bias_log2, cudaStream_t stream);

// One-shot kernel for 129 <= S <= 257 (attention_os.cu): all keys in one N = 256 tcgen05.mma, exact two-pass softmax in
// TMEM, P fed to the P V product straight from TMEM.  mask: MASK_NONE or MASK_KEYLEN; it takes no relative bias.
bool os_supported(int S, int mask);
int launch_os(const __nv_bfloat16* qkv, __nv_bfloat16* out, int B, int S, int W, int H, int mask, const int32_t* kv_len,
              cudaStream_t stream);

}  // namespace attention
}  // namespace mb
