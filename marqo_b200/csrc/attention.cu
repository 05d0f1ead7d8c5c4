#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "attention.cuh"

namespace mb {
namespace attention {

int relative_position_bucket(int d) {
    // MPNetEncoder.relative_position_bucket(d, num_buckets=32, max_distance=128): n = -d; keys after the query take
    // the upper half; |n| < 8 is exact, larger distances are log-spaced up to 128, with torch's fp32 arithmetic
    int ret = 0;
    int n = -d;
    if (n < 0) ret += REL_BUCKETS / 2;
    n = std::abs(n);
    constexpr int max_exact = REL_BUCKETS / 4;   // 8
    if (n < max_exact) return ret + n;
    const float v = std::log((float)n / (float)max_exact) / (float)std::log(128.0 / max_exact) *
                    (float)(REL_BUCKETS / 2 - max_exact);
    return ret + std::min(max_exact + (int)v, REL_BUCKETS / 2 - 1);
}

void fold_relative_bias(const float* rel_bias, int H, int max_dist, float* bias_log2) {
    for (int d = -max_dist; d <= max_dist; ++d) {
        const int dc = std::min(std::max(d, -REL_D), REL_D);
        if (relative_position_bucket(d) != relative_position_bucket(dc))
            fail(B200_ERR_INTERNAL, "relative bias: distance %d is not in the bucket of %d", d, dc);
    }
    for (int h = 0; h < H; ++h)
        for (int d = -REL_D; d <= REL_D; ++d)
            bias_log2[(size_t)h * REL_T + d + REL_D] =
                (float)((double)rel_bias[(size_t)relative_position_bucket(d) * H + h] * 1.4426950408889634);
}

int launch(const __nv_bfloat16* qkv, __nv_bfloat16* out, int B, int S, int W, int H, int mask, const int32_t* kv_len,
           const float* bias_log2, cudaStream_t stream) {
    if (B <= 0 || S <= 0) return 0;
    // A relative-position bias runs on the block kernel only (the one-shot kernel takes none).  Every other length
    // outside the one-shot kernel's range also runs on the block kernel (attention_tc.cu); sequences shorter than one
    // 128-row tile are packed several to a tile under a block-diagonal mask.
    if (bias_log2 == nullptr && os_supported(S, mask)) return launch_os(qkv, out, B, S, W, H, mask, kv_len, stream);
    return launch_tc(qkv, out, B, S, W, H, mask, kv_len, bias_log2, stream);
}

}  // namespace attention
}  // namespace mb
