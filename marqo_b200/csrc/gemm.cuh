// Persistent warp-specialised tcgen05 GEMM:  out[M,N] = epilogue( A[M,K] (bf16, K-major) x W[N,K]^T (bf16, K-major) )
// CTA pairs (cta_group::2): one tcgen05.mma covers a 256 x BN tile across the two SMs of a cluster, each SM holding
// 128 rows of A and BN/2 rows of W; fp32 accumulation in TMEM; TMA-fed 128B-swizzled smem ring (5-6 stages of 32 KB);
// double-buffered accumulators so the 8-warp epilogue of tile i overlaps the MMAs of tile i+1.
#pragma once
#include "common.cuh"

namespace mb {
namespace gemm {

enum Act { ACT_NONE = 0, ACT_GELU = 1, ACT_QUICKGELU = 2 };

struct Epilogue {
    const float* bias = nullptr;      // [N]
    const float* residual = nullptr;  // fp32 [M, ldr], added after the activation
    int ldr = 0;
    int act = ACT_NONE;
    void* out = nullptr;  // bf16 or fp32 [*, ldo]
    int ldo = 0;
    int out_fp32 = 0;
    // ViT token assembly (patch-embed): GEMM row r = (image b, patch i) with G patches per image is written to token
    // row b * (G + 1) + 1 + i and gets rowbias[(1 + i), :] (the positional embedding) added.
    int remap_group = 0;
    const float* rowbias = nullptr;  // fp32 [G + 1, N]
};

// A: bf16 [M, K] row-major with leading dimension lda (elements); W: bf16 [N, K] row-major (nn.Linear layout).
// Requirements: K % 64 == 0, N % 32 == 0, lda % 8 == 0.
void launch(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, int M, int N, int K, const Epilogue& ep,
            int sm_count, cudaStream_t stream);

// ViT patch embedding straight from uint8 pixels (SURVEY §8 a2; add_docs.py:129-134 + clip_utils.py:48-67 fused into the
// conv1 GEMM's operand load): out = epilogue( patches(img) x Wg^T ), where row r of the virtual A matrix is patch r of the
// uint8 HWC batch [n, S, S, 3] (image r / g^2, row-major in the g x g grid), normalised as ToTensor + Normalize, and
// Wg [N, patch_gather_k(patch)] is conv1.weight re-laid by kernels::patch_weight_rows.  No patch matrix exists in HBM:
// the gather warps of the GEMM read the image rows (16-byte coalesced), convert and write the swizzled smem A stage.
struct PatchGather {
    const uint8_t* img = nullptr;
    int n = 0, S = 0, patch = 0;
    float mean[3] = {0.f, 0.f, 0.f}, std[3] = {1.f, 1.f, 1.f};
};
bool patch_gather_supported(int S, int patch);   // S % patch == 0, patch even, 3*S % 16 == 0, S <= 224, grid >= 7
inline int patch_gather_kbpd(int patch) { return (3 * patch + 63) / 64; }
inline int patch_gather_k(int patch) { return patch * patch_gather_kbpd(patch) * 64; }
void launch_patch_embed(const PatchGather& pg, const __nv_bfloat16* Wg, int N, const Epilogue& ep, int sm_count,
                        cudaStream_t stream);

void configure();  // one-time cudaFuncSetAttribute calls

}  // namespace gemm
}  // namespace mb
