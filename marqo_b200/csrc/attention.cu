#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "attention.cuh"

namespace mb {
namespace attention {

constexpr int HD = 64;        // head dim
constexpr int BQ = 64;        // query rows per CTA (4 warps x 16)
constexpr int BKV = 64;       // keys per block
constexpr int THREADS = 128;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void cp_async16(void* dst, const void* src, bool valid) {
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
                 "{%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

// tile: 64 rows x 64 bf16 (128 B per row), 16-byte chunks XOR-swizzled by (row & 7)
__device__ __forceinline__ __nv_bfloat16* tile_ptr(__nv_bfloat16* tile, int row, int chunk) {
    return tile + row * HD + ((chunk ^ (row & 7)) << 3);
}

__device__ __forceinline__ void load_tile(__nv_bfloat16* tile, const __nv_bfloat16* base, int row0, int nrows, int ld) {
    // base points at (sequence row 0, first column of this head's q/k/v slice)
#pragma unroll
    for (int i = 0; i < (64 * 8) / THREADS; ++i) {
        const int idx = threadIdx.x + i * THREADS;
        const int r = idx >> 3, c = idx & 7;
        const bool ok = row0 + r < nrows;
        const __nv_bfloat16* src = base + (size_t)(ok ? row0 + r : 0) * ld + c * 8;
        cp_async16(tile_ptr(tile, r, c), src, ok);
    }
}

template <int MASK>
__global__ void __launch_bounds__(THREADS)
attention_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out, int S, int W,
                 const int32_t* __restrict__ kv_len, float scale_log2e) {
    __shared__ __align__(128) __nv_bfloat16 sQ[BQ * HD];
    __shared__ __align__(128) __nv_bfloat16 sK[2][BKV * HD];
    __shared__ __align__(128) __nv_bfloat16 sV[2][BKV * HD];

    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * BQ;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int ld = 3 * W;
    const __nv_bfloat16* seq = qkv + (size_t)b * S * ld;
    const __nv_bfloat16* qbase = seq + h * HD;
    const __nv_bfloat16* kbase = seq + W + h * HD;
    const __nv_bfloat16* vbase = seq + 2 * W + h * HD;

    int len = S;
    if (MASK == MASK_KEYLEN) len = min(S, max(kv_len[b], 0));
    int kend = len;
    if (MASK == MASK_CAUSAL) kend = min(len, q0 + BQ);
    const int nkb = (kend + BKV - 1) / BKV;

    load_tile(sQ, qbase, q0, S, ld);
    if (nkb > 0) {
        load_tile(sK[0], kbase, 0, len, ld);
        load_tile(sV[0], vbase, 0, len, ld);
    }
    cp_async_commit();

    uint32_t qf[4][4];
    float o[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
    float row_max[2] = {-INFINITY, -INFINITY};
    float row_sum[2] = {0.f, 0.f};
    const int qrow[2] = {q0 + warp * 16 + g, q0 + warp * 16 + g + 8};

    for (int kb = 0; kb < nkb; ++kb) {
        const int buf = kb & 1;
        if (kb + 1 < nkb) {
            load_tile(sK[buf ^ 1], kbase, (kb + 1) * BKV, len, ld);
            load_tile(sV[buf ^ 1], vbase, (kb + 1) * BKV, len, ld);
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        if (kb == 0) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const int mat = lane >> 3, r = lane & 7;
                ldmatrix_x4(qf[ks], tile_ptr(sQ, warp * 16 + (mat & 1) * 8 + r, ks * 2 + (mat >> 1)));
            }
        }
        // ---- S = Q K^T (16 x 64 per warp)
        float s[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int np = 0; np < 4; ++np) {
                uint32_t kf[4];
                const int mat = lane >> 3, r = lane & 7;
                ldmatrix_x4(kf, tile_ptr(sK[buf], np * 16 + (mat >> 1) * 8 + r, ks * 2 + (mat & 1)));
                mma_bf16(s[2 * np], qf[ks], kf[0], kf[1]);
                mma_bf16(s[2 * np + 1], qf[ks], kf[2], kf[3]);
            }
        }
        // ---- mask, scale (log2 domain), online softmax
        float mx[2] = {row_max[0], row_max[1]};
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int key = kb * BKV + nt * 8 + 2 * t + (e & 1);
                const int rr = e >> 1;
                bool ok = key < len;
                if (MASK == MASK_CAUSAL) ok = ok && key <= qrow[rr];
                const float v = ok ? s[nt][e] * scale_log2e : -INFINITY;
                s[nt][e] = v;
                mx[rr] = fmaxf(mx[rr], v);
            }
        }
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            mx[rr] = fmaxf(mx[rr], __shfl_xor_sync(0xffffffffu, mx[rr], 1));
            mx[rr] = fmaxf(mx[rr], __shfl_xor_sync(0xffffffffu, mx[rr], 2));
        }
        float corr[2], msafe[2];
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            msafe[rr] = mx[rr] == -INFINITY ? 0.f : mx[rr];
            corr[rr] = exp2f(row_max[rr] - msafe[rr]);  // row_max = -inf on the first block -> 0
            row_max[rr] = mx[rr];
            row_sum[rr] *= corr[rr];
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            o[nt][0] *= corr[0];
            o[nt][1] *= corr[0];
            o[nt][2] *= corr[1];
            o[nt][3] *= corr[1];
        }
        float ps[2] = {0.f, 0.f};
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float pv = exp2f(s[nt][e] - msafe[e >> 1]);
                s[nt][e] = pv;
                ps[e >> 1] += pv;
            }
        }
        row_sum[0] += ps[0];
        row_sum[1] += ps[1];
        // ---- O += P V
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            uint32_t pa[4];
            pa[0] = pack2(s[2 * ks][0], s[2 * ks][1]);
            pa[1] = pack2(s[2 * ks][2], s[2 * ks][3]);
            pa[2] = pack2(s[2 * ks + 1][0], s[2 * ks + 1][1]);
            pa[3] = pack2(s[2 * ks + 1][2], s[2 * ks + 1][3]);
#pragma unroll
            for (int dp = 0; dp < 4; ++dp) {
                uint32_t vf[4];
                const int mat = lane >> 3, r = lane & 7;
                ldmatrix_x4_trans(vf, tile_ptr(sV[buf], ks * 16 + (mat & 1) * 8 + r, dp * 2 + (mat >> 1)));
                mma_bf16(o[2 * dp], pa, vf[0], vf[1]);
                mma_bf16(o[2 * dp + 1], pa, vf[2], vf[3]);
            }
        }
        __syncthreads();
    }
    if (nkb == 0) {
        cp_async_wait<0>();
        __syncthreads();
    }
    // ---- finalise: O /= rowsum (quad-reduced), stage through sQ (this warp's 16 rows), 16-byte coalesced stores
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
        row_sum[rr] += __shfl_xor_sync(0xffffffffu, row_sum[rr], 1);
        row_sum[rr] += __shfl_xor_sync(0xffffffffu, row_sum[rr], 2);
    }
    const float inv[2] = {row_sum[0] > 0.f ? 1.f / row_sum[0] : 0.f, row_sum[1] > 0.f ? 1.f / row_sum[1] : 0.f};
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        const int r0 = warp * 16 + g;
        *reinterpret_cast<uint32_t*>(tile_ptr(sQ, r0, nt) + 2 * t) = pack2(o[nt][0] * inv[0], o[nt][1] * inv[0]);
        *reinterpret_cast<uint32_t*>(tile_ptr(sQ, r0 + 8, nt) + 2 * t) = pack2(o[nt][2] * inv[1], o[nt][3] * inv[1]);
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int idx = lane + i * 32;
        const int r = warp * 16 + (idx >> 3), c = idx & 7;
        const int tok = q0 + r;
        if (tok < S) {
            const uint4 val = *reinterpret_cast<const uint4*>(tile_ptr(sQ, r, c));
            *reinterpret_cast<uint4*>(out + ((size_t)b * S + tok) * W + h * HD + c * 8) = val;
        }
    }
}

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
    // A relative-position bias runs on the tcgen05 kernel only (the one-shot kernel and the mma.sync kernel take none)
    if (bias_log2) return launch_tc(qkv, out, B, S, W, H, mask, kv_len, bias_log2, stream);
    // Every sequence length runs on the tcgen05 kernel (attention_tc.cu); sequences shorter than one 128-row tile are
    // packed several to a tile under a block-diagonal mask.  MARQO_B200_ATTN_SHORT=mma selects the warp-level
    // mma.sync kernel below for S < 128 (kept for A/B timing only).
    static const bool short_on_mma = [] {
        const char* e = getenv("MARQO_B200_ATTN_SHORT");
        return e != nullptr && strcmp(e, "mma") == 0;
    }();
    if (os_supported(S, mask)) return launch_os(qkv, out, B, S, W, H, mask, kv_len, stream);
    if (S >= 128 || !short_on_mma) {
        return launch_tc(qkv, out, B, S, W, H, mask, kv_len, nullptr, stream);
    }
    if (W != H * HD) fail(B200_ERR_UNSUPPORTED, "attention: head_dim must be 64 (width %d, heads %d)", W, H);
    const dim3 grid((S + BQ - 1) / BQ, H, B);
    const float scale_log2e = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) * log2(e)
    switch (mask) {
        case MASK_NONE:
            attention_kernel<MASK_NONE><<<grid, THREADS, 0, stream>>>(qkv, out, S, W, kv_len, scale_log2e);
            break;
        case MASK_CAUSAL:
            attention_kernel<MASK_CAUSAL><<<grid, THREADS, 0, stream>>>(qkv, out, S, W, kv_len, scale_log2e);
            break;
        case MASK_KEYLEN:
            if (!kv_len) fail(B200_ERR_INTERNAL, "attention: kv_len required for key-length masking");
            attention_kernel<MASK_KEYLEN><<<grid, THREADS, 0, stream>>>(qkv, out, S, W, kv_len, scale_log2e);
            break;
        default:
            fail(B200_ERR_INTERNAL, "attention: unknown mask mode %d", mask);
    }
    MB_CUDA(cudaGetLastError());
    return 1;
}

}  // namespace attention
}  // namespace mb
