#include "gemm.cuh"

#include <mutex>

#include "ptx.cuh"

namespace mb {
namespace gemm {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int UMMA_K = 16;
// Epilogue warps (warp 0 TMA, warp 1 MMA, warps 2.. epilogue):
//   EW = 8   general epilogue (fp32 / residual / token scatter): two warps per TMEM sub-partition, each draining one
//            half of the tile's columns through a 32 x 128 B transpose buffer.
//   EW = 16  bf16-out GEMMs without residual (QKV, fc1 + GELU): FOUR warps per sub-partition, a quarter of the columns
//            each.  The r01 profile of fc1 showed the 8-warp epilogue at 49 % issue-active with two warps per scheduler
//            (31 % of their stall samples fixed-latency dependencies, 16 % tcgen05.ld waits) while the tensor pipe idled
//            at 62 %: the erf-GELU epilogue took as long as the tile's MMAs.  Twice the warps = twice the independent
//            instruction streams per scheduler to hide those latencies; the staging buffer shrinks to 32 x 64 B per
//            warp so the smem ring keeps its depth.
constexpr int ACC_STAGES = 2;
constexpr uint32_t A_STAGE_BYTES = BM * BK * 2;
constexpr int SMEM_LIMIT = 232448;

// GATHER (ViT patch-embed, SURVEY §8 a2): the A operand is not a matrix in HBM.  Four extra warps read the uint8 HWC
// images (whole 16-byte units of the image rows a warp's 32 patches touch, coalesced), stage them in a private smem
// strip, apply ToTensor + Normalize and write bf16 straight into the 128B-swizzled A stage the tensor core reads;
// W (one 64-slot k-block group per patch pixel row, zero padded) still arrives by TMA.
constexpr int GATHER_WARPS = 4;
constexpr int GATHER_MAX_ROWS = 6;          // image-row strips one warp's 32 consecutive patches can touch (grid >= 7)
constexpr int GATHER_MAX_ROW_BYTES = 672;   // 3 * 224
constexpr uint32_t GATHER_WARP_BYTES = 4096;
static_assert(GATHER_MAX_ROWS * GATHER_MAX_ROW_BYTES <= (int)GATHER_WARP_BYTES, "raw strip buffer");

template <int BN, int EW, bool GATHER = false>
struct Cfg {
    static constexpr int THREADS = 64 + 32 * EW + (GATHER ? 32 * GATHER_WARPS : 0);
    static constexpr uint32_t RAW_BYTES = GATHER ? GATHER_WARPS * GATHER_WARP_BYTES : 0;
    static constexpr uint32_t B_STAGE_BYTES = (BN / 2) * BK * 2;   // each CTA of the pair holds half of the W tile
    static constexpr uint32_t STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
    // per epilogue warp: a 32-row transpose buffer (128-byte rows; 64-byte rows for EW = 16) + a 128-byte bias row
    static constexpr uint32_t EPI_ROW_BYTES = EW == 16 ? 64 : 128;
    // (EW = 16 keeps the bias row inside the transpose buffer, so the smem ring stays 6 stages deep at BN = 256)
    // (+ for the general epilogue of a GEMM that can have a residual input: a second 32 x 128 B buffer the NEXT chunk's
    //  residual block is prefetched into with cp.async while the current chunk is processed)
    // Both buffers are 4 KB and 1024-byte aligned: TMA's hardware 128B swizzle (residual in, fp32 result out) works on
    // absolute shared-memory address bits, and must coincide with the epilogue's own (16-byte unit ^ (row & 7)) pattern.
    static constexpr uint32_t RES_BYTES = (EW == 8 && !GATHER) ? 32 * 128 : 0;
    static constexpr uint32_t EPI_WARP_BYTES = 32 * EPI_ROW_BYTES + ((EW == 16 || !GATHER) ? 0 : 128) + RES_BYTES;
    static constexpr uint32_t EPI_BYTES = EW * EPI_WARP_BYTES;
    static constexpr int STAGES_RAW = (SMEM_LIMIT - 2048 - (int)EPI_BYTES - (int)RAW_BYTES) / (int)STAGE_BYTES;
    static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
    static constexpr size_t SMEM_BYTES =
        (size_t)STAGES * STAGE_BYTES + EPI_BYTES + RAW_BYTES + 1024 /*align*/ + 512 /*barriers*/;
    static constexpr uint32_t TMEM_COLS = ACC_STAGES * BN < 32 ? 32 : ACC_STAGES * BN;
};

// CTA pairs (cta_group::2): one tcgen05.mma spans both SMs of a pair — a 256 x BN tile, 128 rows of A and BN/2 rows
// of W in each SM's shared memory.  Per SM and k-block the tensor core reads 16 KB instead of 24 KB and TMA writes
// 32 KB instead of 48 KB, which takes the single-CTA kernel off its shared-memory-bandwidth ceiling (ncu: the MMA
// warp never waited for data, yet the tensor pipe stalled at ~70 %).
constexpr int CLUSTER = 2;

struct Params {
    int M, N, K;
    int tiles_m, tiles_n;   // tiles_m counts 128-row blocks
    int super_m;            // ceil(tiles_m / CLUSTER)
    Epilogue ep;
    int tma_io;             // fp32 output / residual blocks through TMA (tmap_o / tmap_r are valid)
    // GATHER only: uint8 HWC images [n, S, S, 3]; A row r = patch r (image r / (g*g), then row-major in the grid)
    const uint8_t* img;
    int g;                  // patches per image side
    int patch;              // patch edge in pixels
    int row_bytes;          // 3 * S
    int seg;                // 3 * patch: bytes (= k values) of one patch pixel row
    int kbpd;               // 64-slot k-blocks per patch pixel row: ceil(seg / 64)
    int last_steps;         // UMMA_K steps of the last k-block of a pixel row: ceil((seg - 64 (kbpd-1)) / 16)
    float nscale[3], nshift[3];   // (u8 * nscale[c] + nshift[c]) == (u8/255 - mean[c]) / std[c]
};

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// erf(a) = sign(a) * (1 - exp(P(|a|))) with the single-branch minimax polynomial of the large-argument branch of the
// usual float erf (coefficients pre-multiplied by log2(e) so the exponential is one ex2.approx).  Max abs error of
// erf 1.9e-5, of GELU 1.9e-6 (5.9e-5 relative) — two orders below the bf16 rounding applied to the result
// (tests/test_kernels_gpu.py::test_gemm_epilogues compares against torch's exact erf GELU).
__device__ __forceinline__ float gelu_erf(float x) {
    const float a = x * 0.70710678118654752440f;
    const float t = fabsf(a);
    const float s = a * a;
    float r = fmaf(-2.49374837e-5f, t, 5.52836593e-4f);
    const float u = fmaf(-5.60337594e-3f, t, 3.49920232e-2f);
    r = fmaf(r, s, u);
    r = fmaf(r, t, -1.54047912e-1f);
    r = fmaf(r, t, -9.15890168e-1f);
    r = fmaf(r, t, -1.85700115e-1f);
    r = fmaf(r, t, -1.44269504f * t);
    const float e = copysignf(1.0f - ex2_approx(r), a);
    const float hx = 0.5f * x;
    return fmaf(hx, e, hx);
}

// The same erf-GELU on TWO elements per instruction (HFMA2 / ex2.approx.f16x2), for outputs that are rounded to bf16 anyway
// (fc1's epilogue: the r02 profile had it at 16 fp32 instructions per element and the GEMM epilogue-bound at 75 % tensor
// pipe).  fp16 has 11 significand bits against bf16's 8: the result carries ~1e-3 relative error before the bf16 rounding
// of 4e-3 (tests/test_kernels_gpu.py::test_gemm_epilogues; the reference's own CUDA path evaluates GELU in fp16 under
// torch.autocast, open_clip_model.py:256-258).  |x| up to 360 keeps a * a inside fp16 range.
__device__ __forceinline__ __half2 gelu_erf_h2(__half2 x) {
    const __half2 a = __hmul2(x, __float2half2_rn(0.70710678118654752440f));
    const __half2 t = __habs2(a);
    const __half2 s = __hmul2(a, a);
    __half2 r = __hfma2(__float2half2_rn(-2.49374837e-5f), t, __float2half2_rn(5.52836593e-4f));
    const __half2 u = __hfma2(__float2half2_rn(-5.60337594e-3f), t, __float2half2_rn(3.49920232e-2f));
    r = __hfma2(r, s, u);
    r = __hfma2(r, t, __float2half2_rn(-1.54047912e-1f));
    r = __hfma2(r, t, __float2half2_rn(-9.15890168e-1f));
    r = __hfma2(r, t, __float2half2_rn(-1.85700115e-1f));
    r = __hfma2(r, t, __hmul2(t, __float2half2_rn(-1.44269504f)));
    const __half2 e = h2exp2(r);
    const __half2 om = __hsub2(__float2half2_rn(1.0f), e);
    // copysign(1 - e, a) on both halves
    const uint32_t eb = (*reinterpret_cast<const uint32_t*>(&om) & 0x7fff7fffu) | (*reinterpret_cast<const uint32_t*>(&a) & 0x80008000u);
    const __half2 erfv = *reinterpret_cast<const __half2*>(&eb);
    const __half2 hx = __hmul2(x, __float2half2_rn(0.5f));
    return __hfma2(hx, erfv, hx);
}

__device__ __forceinline__ float quick_gelu(float x) {   // x * sigmoid(1.702 x)
    return x / (1.0f + ex2_approx(-1.702f * 1.44269504f * x));
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

// Explicit shared-space accesses for the epilogue's staging buffers: through generic pointers the compiler emitted generic
// LD / ST plus 64-bit address arithmetic (the r02 profile of out_proj: 519 always-executed instructions per 32-column chunk, of
// which 64 FADD, 24 loads and 17 stores were the work).
__device__ __forceinline__ float4 lds_f4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint4 lds_u4(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_f4(uint32_t a, float x, float y, float z, float w) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ void sts_u4(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}

template <int BN, int EW, bool GATHER>
__global__ void __launch_bounds__(64 + 32 * EW + (GATHER ? 32 * GATHER_WARPS : 0), 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
            const __grid_constant__ CUtensorMap tmap_o, const __grid_constant__ CUtensorMap tmap_r, Params p) {
    using C = Cfg<BN, EW, GATHER>;
    constexpr int EPI_WARPS = EW;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + (size_t)C::STAGES * A_STAGE_BYTES;
    uint8_t* smem_epi = smem + (size_t)C::STAGES * C::STAGE_BYTES;
    uint8_t* smem_strip = smem_epi + C::EPI_BYTES;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_strip + C::RAW_BYTES);
    uint64_t* empty = full + C::STAGES;
    uint64_t* tfull = empty + C::STAGES;
    uint64_t* tempty = tfull + ACC_STAGES;
    uint64_t* res_full = tempty + ACC_STAGES;   // [8] one per epilogue warp: its residual block has landed (TMA)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_full + 8);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const int kblocks = p.K / BK;
    const uint32_t crank = ptx::cluster_ctarank();
    const int cluster_id = blockIdx.x / CLUSTER;
    const int num_clusters = gridDim.x / CLUSTER;
    const int num_super = p.super_m * p.tiles_n;   // (pair of m-blocks) x n-block units, one per cluster step

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmap_a);
        ptx::prefetch_tmap(&tmap_b);
        for (int i = 0; i < C::STAGES; ++i) {
            // leader's copy is used: its own arrive.expect_tx + the peer's arrive (+ every gather warp of the pair)
            ptx::mbar_init(&full[i], CLUSTER + (GATHER ? CLUSTER * GATHER_WARPS : 0));
            ptx::mbar_init(&empty[i], 1);         // one multicast tcgen05.commit per use, in each CTA
        }
        for (int i = 0; i < 8; ++i) ptx::mbar_init(&res_full[i], 1);
        for (int i = 0; i < ACC_STAGES; ++i) {
            ptx::mbar_init(&tfull[i], 1);
            ptx::mbar_init(&tempty[i], CLUSTER * EPI_WARPS);   // leader's copy: epilogue warps of both CTAs
        }
        ptx::fence_barrier_init();
    }
    if (warp == 1) {   // executed by both CTAs of the pair
        ptx::tmem_alloc_2sm<C::TMEM_COLS>(tmem_slot);
        ptx::tmem_relinquish_2sm();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();   // the peer's barriers are initialised before any multicast can land there
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int t = cluster_id; t < num_super; t += num_clusters) {
                const int m0 = ((t / p.tiles_n) * CLUSTER + (int)crank) * BM;
                const int n0 = (t % p.tiles_n) * BN;
                for (int kb = 0; kb < kblocks; ++kb) {
                    ptx::mbar_wait(&empty[stage], phase ^ 1);
                    // completion of BOTH CTAs' loads is tracked by the leader's full barrier
                    const uint32_t leader_full = ptx::mapa_u32(ptx::smem_u32(&full[stage]), 0);
                    if (crank == 0)
                        ptx::mbar_arrive_expect_tx(&full[stage], CLUSTER * (GATHER ? C::B_STAGE_BYTES : C::STAGE_BYTES));
                    else
                        ptx::mbar_arrive_cluster(leader_full);
                    if (!GATHER)
                        ptx::tma_load_2d_2sm(smem_a + (size_t)stage * A_STAGE_BYTES, &tmap_a, leader_full, kb * BK, m0,
                                             ptx::kEvictNormal);
                    ptx::tma_load_2d_2sm(smem_b + (size_t)stage * C::B_STAGE_BYTES, &tmap_b, leader_full, kb * BK,
                                         n0 + (int)crank * (BN / CLUSTER), ptx::kEvictLast);
                    if (++stage == C::STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1 && crank == 0) {
        constexpr uint32_t idesc = ptx::make_idesc_f16(1 /*bf16*/, CLUSTER * BM, BN);   // M = 256 across the pair
        int stage = 0, acc = 0;
        uint32_t phase = 0, acc_phase = 0;
        for (int t = cluster_id; t < num_super; t += num_clusters) {
            ptx::mbar_wait(&tempty[acc], acc_phase ^ 1);
            ptx::tc_fence_after();
            for (int kb = 0; kb < kblocks; ++kb) {
                ptx::mbar_wait(&full[stage], phase);
                ptx::tc_fence_after();
                if (lane == 0) {
                    const uint32_t a_base = ptx::smem_u32(smem_a + (size_t)stage * A_STAGE_BYTES);
                    const uint32_t b_base = ptx::smem_u32(smem_b + (size_t)stage * C::B_STAGE_BYTES);
                    // GATHER: the last k-block of a patch pixel row holds fewer than 64 values; the slots past them are
                    // never written by the gather warps, so those UMMA_K steps are not issued
                    const int ksteps = (GATHER && (kb % p.kbpd) == p.kbpd - 1) ? p.last_steps : BK / UMMA_K;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k)
                        if (k < ksteps)
                            ptx::umma_f16_2sm(tmem_base + acc * BN, ptx::make_desc_k_sw128(a_base + k * UMMA_K * 2),
                                              ptx::make_desc_k_sw128(b_base + k * UMMA_K * 2), idesc,
                                              (kb | k) != 0 ? 1u : 0u);
                    // both CTAs' producers get their stage back; both CTAs' epilogues get the finished accumulator
                    ptx::umma_commit_2sm(&empty[stage], (uint16_t)((1u << CLUSTER) - 1));
                    if (kb == kblocks - 1) ptx::umma_commit_2sm(&tfull[acc], (uint16_t)((1u << CLUSTER) - 1));
                }
                __syncwarp();
                if (++stage == C::STAGES) {
                    stage = 0;
                    phase ^= 1;
                }
            }
            if (++acc == ACC_STAGES) {
                acc = 0;
                acc_phase ^= 1;
            }
        }
    } else if (warp >= 2 && warp < 2 + EW && EW == 16) {
        // ---------------------------------------------------------------- fast bf16 epilogue (16 warps)
        // lane == accumulator row; each warp drains 32 rows x (BN / 4) columns in 32-column chunks:
        // bias -> activation -> bf16 -> 32 x 64 B swizzled staging buffer -> 64-byte coalesced row segments.
        const int sp = warp & 3;
        const int part = (warp - 2) >> 2;                  // column quarter of the tile
        constexpr int PART_COLS = BN / 4;
        constexpr int CHUNKS = PART_COLS / 32;
        static_assert(EW != 16 || (BN % 128 == 0), "the 16-warp epilogue needs whole 32-column chunks per quarter");
        const Epilogue& ep = p.ep;
        uint8_t* stage_buf = smem_epi + (size_t)(warp - 2) * C::EPI_WARP_BYTES;
        float* bias_row = reinterpret_cast<float*>(stage_buf);   // first 128 B of the buffer, consumed before it is filled
        const int frow = lane >> 2, funit = lane & 3;      // flush phase: 8 rows x 4 sixteen-byte units per instruction
        const int wswz = (lane >> 1) & 3;                  // write-phase swizzle of this lane's own row
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int t = cluster_id; t < num_super; t += num_clusters) {
            const int m0 = ((t / p.tiles_n) * CLUSTER + (int)crank) * BM;
            const int nt0 = (t % p.tiles_n) * BN + part * PART_COLS;
            const int wrow0 = m0 + sp * 32;
            ptx::mbar_wait(&tfull[acc], acc_phase);
            ptx::tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < CHUNKS; ++c) {
                const int n0 = nt0 + c * 32;
                const bool cols_ok = n0 < p.N;
                float bias_v = 0.f;
                if (ep.bias && cols_ok) bias_v = __ldg(ep.bias + n0 + lane);
                uint32_t v[32];
                ptx::tmem_ld_32x32b_x32(tmem_base + (uint32_t(sp * 32) << 16) + acc * BN + part * PART_COLS + c * 32, v);
                ptx::tmem_ld_wait();
                if (c == CHUNKS - 1) {
                    // this warp's share of the accumulator is in registers: hand it back to the MMA warp
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa_u32(ptx::smem_u32(&tempty[acc]), 0));
                }
                if (cols_ok) {
                    bias_row[lane] = bias_v;
                    __syncwarp();
                    float f[32];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float4 b = *reinterpret_cast<const float4*>(bias_row + 4 * j);   // broadcast read
                        f[4 * j] = __uint_as_float(v[4 * j]) + b.x;
                        f[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + b.y;
                        f[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + b.z;
                        f[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + b.w;
                    }
                    __syncwarp();   // every lane has read the bias row: the buffer may be overwritten
                    // one uniform branch per chunk, NOT a per-element select: with `apply_act(f, ep.act)` inside the loop
                    // the compiler if-converted the switch and every element paid for erf-GELU AND QuickGELU (two ex2 and
                    // a reciprocal, ~40 instructions per element in the r02 SASS; fc1 was epilogue-bound at 73 % tensor pipe)
                    uint32_t pk[16];
                    if (ep.act == ACT_GELU) {
                        // packed-half erf-GELU: two elements per instruction
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float2 y = __half22float2(gelu_erf_h2(__floats2half2_rn(f[2 * j], f[2 * j + 1])));
                            pk[j] = pack_bf16x2(y.x, y.y);
                        }
                    } else {
                        if (ep.act == ACT_QUICKGELU) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) f[j] = quick_gelu(f[j]);
                        }
#pragma unroll
                        for (int j = 0; j < 16; ++j) pk[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<uint4*>(stage_buf + lane * 64 + ((j ^ wswz) << 4)) =
                            make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                    __syncwarp();
                    const int col = n0 + funit * 8;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int rr = i * 8 + frow;
                        const int grow = wrow0 + rr;
                        if (grow < p.M) {
                            const uint4 val = *reinterpret_cast<const uint4*>(stage_buf + rr * 64 + ((funit ^ ((rr >> 1) & 3)) << 4));
                            *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(ep.out) + ((size_t)grow * ep.ldo + col) * 2) = val;
                        }
                    }
                    __syncwarp();   // the buffer (and bias_row) are reused by the next chunk
                }
            }
            if (++acc == ACC_STAGES) {
                acc = 0;
                acc_phase ^= 1;
            }
        }
    } else if (warp >= 2 && warp < 2 + EW) {
        // ---------------------------------------------------------------- epilogue (TMEM -> regs -> smem -> global)
        // A warp may only read the TMEM lanes of sub-partition (warp % 4); the two warps that share a sub-partition
        // split the tile's columns in halves, so 8 warps drain one 128 x BN accumulator.  TMEM hands every lane one ROW
        // (32 consecutive columns); global memory wants whole 128-byte lines per instruction, so each warp transposes
        // through a private, XOR-swizzled 32 x 128 B shared-memory buffer in both directions (residual in, result out).
        const int sp = warp & 3;
        const int half = (warp - 2) >> 2;
        constexpr int HALF_COLS = BN / 2 >= 32 ? BN / 2 : 32;
        constexpr int CHUNKS = HALF_COLS / 32;
        const bool has_cols = half * HALF_COLS < BN;  // BN = 32 would leave the second half empty
        const Epilogue& ep = p.ep;
        const float* const residual = GATHER ? nullptr : ep.residual;   // the patch-embed GEMM has no residual input
        uint8_t* stage_buf = smem_epi + (size_t)(warp - 2) * C::EPI_WARP_BYTES;
        uint8_t* res_buf = stage_buf + 32 * 128 + (GATHER ? 128 : 0);   // residual block of the chunk about to be processed
        // fp32 results without token remap leave through TMA (one bulk tensor store per 32 x 32 block instead of 8 shared
        // loads + 8 global stores + their address arithmetic per lane), residual blocks arrive through TMA: p.tma_io.
        const bool tma_io = !GATHER && p.tma_io != 0;
        uint64_t* my_res_full = &res_full[warp - 2];
        uint32_t res_phase = 0;
        const int esz = ep.out_fp32 ? 4 : 2;                  // output element size
        const int cols_per_flush = 128 / esz;                 // 32 fp32 or 64 bf16 columns fill a 128-byte row
        // bf16 results are staged two chunks (64 columns) per flush; a residual block occupies the whole buffer, so
        // residual GEMMs (fp32 out in this engine) flush after every chunk
        const int chunks_per_flush = (ep.out_fp32 || residual) ? 1 : cols_per_flush / 32;
        const int srow = lane >> 3, sunit = lane & 7;         // coalesced phase: 4 rows x 8 sixteen-byte units per instr
        // Residual blocks travel global -> shared memory asynchronously, one chunk AHEAD of their use (and across the
        // tile boundary: the next tile's first block is requested before this warp waits for that accumulator), in the
        // swizzled layout the lane == row read expects.  The r02 profile had out_proj (K = 1024: a tile every ~7 us) at
        // 44-47 % tensor pipe with its 8 epilogue warps taking one exposed L2 round trip per 32-column chunk.
        // lane-constant shared addresses.  Coalesced phase (4 rows x 8 sixteen-byte units per instruction), row rr = 4 i + srow:
        //   addr(i) = base + rr * 128 + ((sunit ^ (rr & 7)) << 4) = (co_even | co_odd picked by i & 1) + i * 512
        // Row phase (lane == row): addr(j) = (base + lane * 128) | ((j ^ (lane & 7)) << 4) = rowp ^ (j << 4)
        const uint32_t stage_s = ptx::smem_u32(stage_buf), res_s = ptx::smem_u32(res_buf);
        const uint32_t co_even = (uint32_t)(srow * 128 + ((sunit ^ srow) << 4));
        const uint32_t co_odd = co_even ^ 64u;
        const uint32_t rowp = (uint32_t)(lane * 128 + ((lane & 7) << 4));
        int pref_t = -1, pref_c = -1;   // the (tile, chunk) whose residual block is in res_buf / on its way there
        auto prefetch_residual = [&](int tt, int cc) {
            if (GATHER || !residual || !has_cols || tt >= num_super) return;
            const int pm0 = ((tt / p.tiles_n) * CLUSTER + (int)crank) * BM + sp * 32;
            const int pn0 = (tt % p.tiles_n) * BN + half * HALF_COLS + cc * 32;
            if (pn0 >= p.N) return;
            if (tma_io) {
                if (lane == 0) {
                    ptx::mbar_arrive_expect_tx(my_res_full, 32 * 128);
                    ptx::tma_load_2d(res_buf, &tmap_r, my_res_full, pn0, pm0, ptx::kEvictNormal);   // rows >= M: zero fill
                }
                pref_t = tt;
                pref_c = cc;
                return;
            }
            const float* src0 = residual + (size_t)(pm0 + srow) * ep.ldr + pn0 + sunit * 4;   // row slot 0 of this lane
            const size_t step = (size_t)4 * ep.ldr;                                           // next row slot: 4 rows on
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const bool ok = pm0 + i * 4 + srow < p.M;
                const float* src = ok ? src0 + i * step : residual;
                const uint32_t dst = res_s + ((i & 1) ? co_odd : co_even) + i * 512;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(ok ? 16 : 0) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
            pref_t = tt;
            pref_c = cc;
        };
        int acc = 0;
        uint32_t acc_phase = 0;
        prefetch_residual(cluster_id, 0);
        for (int t = cluster_id; t < num_super; t += num_clusters) {
            const int m0 = ((t / p.tiles_n) * CLUSTER + (int)crank) * BM;
            const int nt0 = (t % p.tiles_n) * BN + half * HALF_COLS;
            const int wrow0 = m0 + sp * 32;                   // first row of this warp's 32-row band
            // (not for long K: a tile of fc2, K = 4096, takes ~28 us during which ~80 MB stream through the L2 — the lines
            // were evicted again before their use and the residual was fetched from HBM twice: r01/r02 ncu 1.32 GB per
            // launch against 1.085 GB algorithmic.  Its epilogue has four times the slack to take the HBM latency itself.)
            if (residual && has_cols && p.K <= 2048) {
                // pull the residual band this warp needs for its NEXT tile towards L2 (the very first tile: itself)
                for (int pass = (t == cluster_id ? 0 : 1); pass < 2; ++pass) {
                    const int tn = t + pass * num_clusters;
                    if (tn >= num_super) break;
                    const int prow = ((tn / p.tiles_n) * CLUSTER + (int)crank) * BM + sp * 32 + lane;
                    const int pn0 = (tn % p.tiles_n) * BN + half * HALF_COLS;
                    if (prow < p.M) {
                        const char* r = reinterpret_cast<const char*>(residual + (size_t)prow * ep.ldr + pn0);
#pragma unroll
                        for (int l = 0; l < HALF_COLS * 4 / 128; ++l)
                            if (pn0 + l * 32 < p.N) asm volatile("prefetch.global.L2 [%0];" ::"l"(r + l * 128));
                    }
                }
            }
            ptx::mbar_wait(&tfull[acc], acc_phase);
            ptx::tc_fence_after();
            // per tile: the 8 output rows this lane flushes (element offsets of their first column, validity mask)
            uint32_t ooff[8];
            uint32_t okmask = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int grow = wrow0 + i * 4 + srow;
                long long orow = grow;
                if (ep.remap_group > 0) {
                    const int b = grow / ep.remap_group;
                    orow = (long long)b * (ep.remap_group + 1) + 1 + (grow - b * ep.remap_group);
                }
                ooff[i] = (uint32_t)(orow * ep.ldo);
                okmask |= (grow < p.M ? 1u : 0u) << i;
            }
            uint8_t* const out_base = reinterpret_cast<uint8_t*>(ep.out);
#pragma unroll 1
            for (int c = 0; c < CHUNKS; ++c) {
                const int n0 = nt0 + c * 32;
                const bool cols_ok = has_cols && n0 < p.N;
                // (1) accumulator chunk: lane == row
                uint32_t v[32];
                if (has_cols) {
                    ptx::tmem_ld_32x32b_x32(tmem_base + (uint32_t(sp * 32) << 16) + acc * BN + half * HALF_COLS + c * 32, v);
                    ptx::tmem_ld_wait();
                }
                if (c == CHUNKS - 1) {
                    // this warp's share of the accumulator is in registers: hand it back to the MMA warp
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa_u32(ptx::smem_u32(&tempty[acc]), 0));
                }
                if (cols_ok) {
                    if (residual) {
                        // normally requested one chunk ago; a warp whose previous tile had no columns asks now
                        if (pref_t != t || pref_c != c) prefetch_residual(t, c);
                        if (tma_io) {
                            ptx::mbar_wait(my_res_full, res_phase);
                            res_phase ^= 1;
                        } else {
                            asm volatile("cp.async.wait_group 0;" ::: "memory");
                            __syncwarp();   // every lane's part of the residual block has landed
                        }
                    }
                    float f[32];
                    if (ep.bias) {
                        // the chunk's 32 bias values: the same 128 bytes for every lane (L1 broadcast), no smem round trip
                        const float4* b4 = reinterpret_cast<const float4*>(ep.bias + n0);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float4 b = __ldg(b4 + j);
                            f[4 * j] = __uint_as_float(v[4 * j]) + b.x;
                            f[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + b.y;
                            f[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + b.z;
                            f[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + b.w;
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                    }
                    if (ep.act == ACT_GELU) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) f[j] = gelu_erf(f[j]);
                    } else if (ep.act == ACT_QUICKGELU) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) f[j] = quick_gelu(f[j]);
                    }
                    if (ep.rowbias) {   // ViT patch-embed: positional embedding of this lane's patch
                        const int row = wrow0 + lane;
                        const int brow = 1 + row % ep.remap_group;
                        const float4* r4 = reinterpret_cast<const float4*>(ep.rowbias + (size_t)brow * p.N + n0);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float4 b = __ldg(r4 + j);
                            f[4 * j] += b.x;
                            f[4 * j + 1] += b.y;
                            f[4 * j + 2] += b.z;
                            f[4 * j + 3] += b.w;
                        }
                    }
                    if (residual) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float4 b = lds_f4(res_s + (rowp ^ (uint32_t)(j << 4)));
                            f[4 * j] += b.x;
                            f[4 * j + 1] += b.y;
                            f[4 * j + 2] += b.z;
                            f[4 * j + 3] += b.w;
                        }
                        __syncwarp();   // everyone has read its residual row: request the next block into the same buffer
                        if (c + 1 < CHUNKS) prefetch_residual(t, c + 1);
                        else prefetch_residual(t + num_clusters, 0);
                    }
                    // (2) own row -> staging buffer (swizzled 16-byte units)
                    if (tma_io) {   // the previous block's bulk store must have read the buffer out
                        if (lane == 0) ptx::tma_store_wait_read<0>();
                        __syncwarp();
                    }
                    if (ep.out_fp32) {
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            sts_f4(stage_s + (rowp ^ (uint32_t)(j << 4)), f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                    } else {
                        const int ubase = (c % chunks_per_flush) * 4;   // this chunk fills units 0-3 or 4-7 of the row
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            sts_u4(stage_s + (rowp ^ (uint32_t)((ubase + j) << 4)), pack_bf16x2(f[8 * j], f[8 * j + 1]),
                                   pack_bf16x2(f[8 * j + 2], f[8 * j + 3]), pack_bf16x2(f[8 * j + 4], f[8 * j + 5]),
                                   pack_bf16x2(f[8 * j + 6], f[8 * j + 7]));
                    }
                }
                // (3) flush full 128-byte rows: every instruction writes 4 rows x 128 contiguous bytes
                const bool flush = (c % chunks_per_flush) == chunks_per_flush - 1 || c == CHUNKS - 1;
                if (tma_io) {
                    if (cols_ok && wrow0 < p.M) {
                        ptx::fence_proxy_async_smem();   // generic-proxy staging stores -> visible to the bulk store
                        __syncwarp();
                        if (lane == 0) {
                            ptx::tma_store_2d(&tmap_o, stage_buf, n0, wrow0);   // rows >= M / columns >= N are clipped
                            ptx::tma_store_commit();
                        }
                    }
                } else if (flush && has_cols) {
                    __syncwarp();
                    const int fc0 = nt0 + (c / chunks_per_flush) * chunks_per_flush * 32;   // first column held in the buffer
                    const int col = fc0 + sunit * (16 / esz);
                    const int filled_units = ((c % chunks_per_flush) + 1) * (32 * esz / 16);
                    if (col < p.N && sunit < filled_units) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            if ((okmask >> i) & 1u) {
                                const uint4 val = lds_u4(stage_s + ((i & 1) ? co_odd : co_even) + i * 512);
                                *reinterpret_cast<uint4*>(out_base + (size_t)(ooff[i] + (uint32_t)col) * esz) = val;
                            }
                        }
                    }
                    __syncwarp();
                }
            }
            if (++acc == ACC_STAGES) {
                acc = 0;
                acc_phase ^= 1;
            }
        }
        if (tma_io && lane == 0) ptx::tma_store_wait<0>();
    } else if (GATHER && warp >= 2 + EW) {
        // ---------------------------------------------------------------- patch gather (uint8 HWC -> bf16 A stage)
        // Warp gw owns rows gw*32 .. gw*32+31 of this CTA's 128-row A tile: lane == patch.  Per patch pixel row dy the
        // warp copies the image-row strips its patches lie on (whole rows of 3*S bytes, 16-byte units, coalesced) into its
        // private smem strip buffer, then every lane converts its own 3*patch bytes: k = dy*(64*kbpd) + dx*3 + c.
        const int gw = warp - (2 + EW);
        uint8_t* strip = smem_strip + (size_t)gw * GATHER_WARP_BYTES;
        const int r = gw * 32 + lane;                  // row of the A tile
        const int upr = p.row_bytes >> 4;              // 16-byte units per image row
        const uint32_t leader_full0 = ptx::mapa_u32(ptx::smem_u32(&full[0]), 0);
        int stage = 0;
        uint32_t phase = 0;
        for (int t = cluster_id; t < num_super; t += num_clusters) {
            const int m0 = ((t / p.tiles_n) * CLUSTER + (int)crank) * BM + gw * 32;
            // patches past M (last tile) are clamped to the last real patch: their rows are computed and never stored
            const int pfirst = min(m0, p.M - 1), plast = min(m0 + 31, p.M - 1), pl = min(m0 + lane, p.M - 1);
            const int pr0 = pfirst / p.g;              // global patch-row index = image * g + gy
            const int prl = pl / p.g;
            const int nunits = (plast / p.g - pr0 + 1) * upr;
            const int my_off = (prl - pr0) * p.row_bytes + (pl - prl * p.g) * p.seg;
            // per lane: up to 8 sixteen-byte units of the strips (offset of the dy = 0 row, in 16-byte units)
            uint32_t uoff[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int idx = lane + 32 * i;
                const int rr = idx / upr, uu = idx - rr * upr;
                const int pr = pr0 + rr;
                const int b = pr / p.g, gy = pr - b * p.g;
                uoff[i] = idx < nunits ? (uint32_t)(((size_t)b * (p.g * p.patch) + (size_t)gy * p.patch) * upr + uu) : 0xffffffffu;
            }
            const uint4* img4 = reinterpret_cast<const uint4*>(p.img);
            uint4 pre[8];
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (uoff[i] != 0xffffffffu) pre[i] = __ldg(img4 + uoff[i]);
            for (int dy = 0; dy < p.patch; ++dy) {
                __syncwarp();   // every lane has finished converting the previous pixel row out of the strip buffer
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (uoff[i] != 0xffffffffu) *reinterpret_cast<uint4*>(strip + (size_t)(lane + 32 * i) * 16) = pre[i];
                __syncwarp();
                if (dy + 1 < p.patch) {   // next pixel row's loads fly while this one is converted
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        if (uoff[i] != 0xffffffffu) pre[i] = __ldg(img4 + uoff[i] + (size_t)(dy + 1) * upr);
                }
                for (int j = 0; j < p.kbpd; ++j) {
                    const int nvals = min(64, p.seg - 64 * j);   // k values of this k-block (even: seg is even)
                    const int cj = j % 3;                          // channel of the k-block's first byte: (64 j) % 3
                    float sc[3], sh[3];
#pragma unroll
                    for (int x = 0; x < 3; ++x) {
                        const int c = (x + cj) % 3;
                        sc[x] = p.nscale[c];
                        sh[x] = p.nshift[c];
                    }
                    const uint8_t* src = strip + my_off + 64 * j;
                    ptx::mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t* dst = smem_a + (size_t)stage * A_STAGE_BYTES + (size_t)r * 128;
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (u * 8 < ((nvals + 15) & ~15)) {   // whole UMMA_K steps (zero filled); later ones are never issued
                            float f[8];
#pragma unroll
                            for (int e = 0; e < 8; e += 2) {
                                const int k = u * 8 + e;
                                const uint32_t two = k < nvals ? *reinterpret_cast<const uint16_t*>(src + k) : 0u;
                                f[e] = k < nvals ? fmaf((float)(two & 0xffu), sc[k % 3], sh[k % 3]) : 0.f;
                                f[e + 1] = k < nvals ? fmaf((float)(two >> 8), sc[(k + 1) % 3], sh[(k + 1) % 3]) : 0.f;
                            }
                            *reinterpret_cast<uint4*>(dst + ((u ^ (r & 7)) << 4)) =
                                make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]),
                                           pack_bf16x2(f[6], f[7]));
                        }
                    }
                    ptx::fence_proxy_async_smem();   // generic-proxy stores -> visible to the tensor core's async proxy
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive_cluster(leader_full0 + (uint32_t)stage * 8u);
                    if (++stage == C::STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();   // nobody exits while the peer may still multicast into / arrive on this CTA's smem
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc_2sm<C::TMEM_COLS>(tmem_base);
    }
}

void configure() {
    static std::once_flag once;
    std::call_once(once, [] {
        const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
        MB_CUDA(cudaFuncSetAttribute(gemm_kernel<256, 8, false>, attr, (int)Cfg<256, 8>::SMEM_BYTES));
        MB_CUDA(cudaFuncSetAttribute(gemm_kernel<128, 8, false>, attr, (int)Cfg<128, 8>::SMEM_BYTES));
        MB_CUDA(cudaFuncSetAttribute(gemm_kernel<64, 8, false>, attr, (int)Cfg<64, 8>::SMEM_BYTES));
        MB_CUDA(cudaFuncSetAttribute(gemm_kernel<256, 16, false>, attr, (int)Cfg<256, 16>::SMEM_BYTES));
        MB_CUDA(cudaFuncSetAttribute(gemm_kernel<128, 16, false>, attr, (int)Cfg<128, 16>::SMEM_BYTES));
        MB_CUDA(cudaFuncSetAttribute(gemm_kernel<256, 8, true>, attr, (int)Cfg<256, 8, true>::SMEM_BYTES));
        MB_CUDA(cudaFuncSetAttribute(gemm_kernel<128, 8, true>, attr, (int)Cfg<128, 8, true>::SMEM_BYTES));
    });
}

template <int BN, int EW, bool GATHER = false>
static void launch_bn(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, int M, int N, int K, const Epilogue& ep,
                      int sms, cudaStream_t stream, const PatchGather* pg = nullptr) {
    Params p{};
    if (GATHER) {
        p.img = pg->img;
        p.patch = pg->patch;
        p.g = pg->S / pg->patch;
        p.row_bytes = 3 * pg->S;
        p.seg = 3 * pg->patch;
        p.kbpd = patch_gather_kbpd(pg->patch);
        p.last_steps = (p.seg - 64 * (p.kbpd - 1) + UMMA_K - 1) / UMMA_K;
        for (int c = 0; c < 3; ++c) {
            p.nscale[c] = (float)(1.0 / (255.0 * (double)pg->std[c]));
            p.nshift[c] = (float)(-(double)pg->mean[c] / (double)pg->std[c]);
        }
    }
    p.M = M;
    p.N = N;
    p.K = K;
    p.tiles_m = (M + BM - 1) / BM;
    p.tiles_n = (N + BN - 1) / BN;
    p.super_m = (p.tiles_m + CLUSTER - 1) / CLUSTER;
    p.ep = ep;
    // (GATHER has no A matrix: the A map is a second, unused view of W so the kernel signature stays the same)
    CUtensorMap ta = GATHER ? make_tmap_2d(W, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)K, (uint64_t)N, (uint64_t)K * 2,
                                           BK, BN / CLUSTER, CU_TENSOR_MAP_SWIZZLE_128B)
                            : make_tmap_2d(A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)K, (uint64_t)M,
                                           (uint64_t)lda * 2, BK, BM, CU_TENSOR_MAP_SWIZZLE_128B);
    // each CTA of the pair fetches (and keeps) BN / 2 rows of the W tile
    CUtensorMap tb = make_tmap_2d(W, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)K, (uint64_t)N, (uint64_t)K * 2, BK,
                                  BN / CLUSTER, CU_TENSOR_MAP_SWIZZLE_128B);
    const int max_clusters = sms / CLUSTER;
    const int clusters = std::min(p.super_m * p.tiles_n, max_clusters);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(clusters * CLUSTER);
    cfg.blockDim = dim3(Cfg<BN, EW, GATHER>::THREADS);
    cfg.dynamicSmemBytes = Cfg<BN, EW, GATHER>::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CLUSTER;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    // fp32 output without token remap: the epilogue's 32 x 32 blocks (128-byte rows, 128B swizzle) go through TMA
    p.tma_io = (!GATHER && EW == 8 && ep.out_fp32 && ep.remap_group == 0 && ep.rowbias == nullptr &&
                ep.ldo % 4 == 0 && (ep.residual == nullptr || ep.ldr % 4 == 0) &&
                (reinterpret_cast<uintptr_t>(ep.out) & 15) == 0 && (reinterpret_cast<uintptr_t>(ep.residual) & 15) == 0)
                   ? 1 : 0;
    CUtensorMap to = tb, tr = tb;
    if (p.tma_io) {
        to = make_tmap_2d(ep.out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (uint64_t)N, (uint64_t)M, (uint64_t)ep.ldo * 4, 32, 32,
                          CU_TENSOR_MAP_SWIZZLE_128B);
        if (ep.residual)
            tr = make_tmap_2d(ep.residual, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (uint64_t)N, (uint64_t)M,
                              (uint64_t)ep.ldr * 4, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B);
    }
    MB_CUDA(cudaLaunchKernelEx(&cfg, gemm_kernel<BN, EW, GATHER>, ta, tb, to, tr, p));
}

bool patch_gather_supported(int S, int patch) {
    if (S <= 0 || patch <= 0 || S % patch != 0 || patch % 2 != 0) return false;
    if ((3 * S) % 16 != 0 || 3 * S > GATHER_MAX_ROW_BYTES) return false;
    const int g = S / patch;
    return 31 / g + 2 <= GATHER_MAX_ROWS;   // image-row strips under 32 consecutive patches
}

void launch_patch_embed(const PatchGather& pg, const __nv_bfloat16* Wg, int N, const Epilogue& ep, int sms,
                        cudaStream_t stream) {
    if (pg.n <= 0 || N <= 0) return;
    if (!patch_gather_supported(pg.S, pg.patch))
        fail(B200_ERR_INTERNAL, "patch gather: image %d / patch %d is not supported", pg.S, pg.patch);
    if (N % 32 != 0 || ep.ldo % 8 != 0) fail(B200_ERR_INTERNAL, "patch gather: N = %d, ldo = %d", N, ep.ldo);
    if (ep.residual != nullptr || !ep.out_fp32) fail(B200_ERR_INTERNAL, "patch gather: fp32 output without residual only");
    configure();
    const int g = pg.S / pg.patch;
    const long long M = (long long)pg.n * g * g;
    if (M > 0x7fffffffLL || (long long)pg.n * pg.S * pg.S * 3 / 16 >= 0xffffffffLL)
        fail(B200_ERR_INVALID_ARG, "patch gather: batch of %d images is too large", pg.n);
    const int K = patch_gather_k(pg.patch);
    if (N % 256 == 0 || N > 512) launch_bn<256, 8, true>(nullptr, 0, Wg, (int)M, N, K, ep, sms, stream, &pg);
    else launch_bn<128, 8, true>(nullptr, 0, Wg, (int)M, N, K, ep, sms, stream, &pg);
}

void launch(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, int M, int N, int K, const Epilogue& ep, int sms,
            cudaStream_t stream) {
    if (M <= 0 || N <= 0) return;
    if (K <= 0 || K % BK != 0) fail(B200_ERR_INTERNAL, "gemm: K = %d must be a positive multiple of %d", K, BK);
    if (N % 32 != 0) fail(B200_ERR_INTERNAL, "gemm: N = %d must be a multiple of 32", N);
    if (lda % 8 != 0 || ep.ldo % 8 != 0) fail(B200_ERR_INTERNAL, "gemm: leading dimensions must be multiples of 8");
    {   // the epilogues address the output with 32-bit element offsets
        const long long out_rows = (long long)M + (ep.remap_group > 0 ? M / ep.remap_group + 1 : 0) + 256;
        if (out_rows * ep.ldo >= (1LL << 32)) fail(B200_ERR_UNSUPPORTED, "gemm: output of %lld x %d elements is too large", out_rows, ep.ldo);
    }
    configure();
    // bf16 output, no residual / token scatter (QKV, fc1): the 16-warp epilogue
    const bool fast = !ep.out_fp32 && ep.residual == nullptr && ep.rowbias == nullptr && ep.remap_group == 0;
    // Largest tile that wastes no columns, otherwise the widest one.
    if (N % 256 == 0 || N > 512) {
        if (fast) launch_bn<256, 16>(A, lda, W, M, N, K, ep, sms, stream);
        else launch_bn<256, 8>(A, lda, W, M, N, K, ep, sms, stream);
    } else if (N % 128 == 0 || N > 128) {
        if (fast) launch_bn<128, 16>(A, lda, W, M, N, K, ep, sms, stream);
        else launch_bn<128, 8>(A, lda, W, M, N, K, ep, sms, stream);
    } else {
        launch_bn<64, 8>(A, lda, W, M, N, K, ep, sms, stream);
    }
}

}  // namespace gemm
}  // namespace mb
