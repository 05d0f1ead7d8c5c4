// "One-shot" tcgen05 attention for sequences of 129 .. 257 tokens (ViT-L-14: 257; the headline workload), head_dim 64.
//
// All keys of a sequence fit ONE tcgen05.mma of N = 256, so there is no online softmax: per (batch, head, 128 queries)
//   S = Q K^T        (M = 128, N = 256, K = 64)   -> TMEM columns [0, 256)   one instruction group, one hand-off
//   P = exp2(S * scale - ref) in ONE pass over S in TMEM (ref = the row's first-chunk maximum + 32: any reference gives the
//   same softmax, see the softmax warps), written back INTO TMEM as packed bf16 pairs over the columns of S the pass has
//   already consumed ([0, 128)),
//   O = P V          (M = 128, N = 64, K = 256; A operand read from TMEM, V MN-major from smem) -> columns [128, 192)
//   the 257th token's key (257 = 256 + 1): its K / V rows arrive as 16-row TMA boxes, its scores against the item's 128 rows
//   are a 16-column MMA issued together with P V into columns S no longer needs ([192, 208)),
//   epilogue: O / l with the remainder key folded in (exact online update) -> bf16.
// Compared with attention_tc.cu (128-key blocks, P through shared memory, running maximum + O rescale) an item has one
// S / P / O hand-off instead of two of each, no P stores to shared memory, no fence.proxy.async, no rescale branch, and
// K / V are loaded ONCE per (batch, head) and shared by its two query blocks (Q is double buffered).
// The r02 profile of the block kernel (profiles/r02_ncu_summary.md §3) showed the softmax warps waiting on those
// hand-offs for a third of their time and the tensor pipe at 16 %.
//
// Warp roles (224 threads, two CTAs per SM, 256 TMEM columns each):
//   warp 0  TMA producer: Q tiles (2-deep ring), K and V (256 rows each, one load per (batch, head))
//   warp 1  tcgen05.mma issuer
//   warps 2-5  softmax / epilogue, one thread per query row (TMEM lane == row)
//   warp 6  the remainder QUERY row (mma.sync against the K / V tiles while they sit in shared memory), once per
//           (batch, head), as soon as the tiles have landed
#include <algorithm>
#include <mutex>

#include "attention.cuh"
#include "ptx.cuh"

namespace mb {
namespace attention {
namespace os {

constexpr int HD = 64;
constexpr int BQ = 128;
constexpr int NK = 256;                       // keys covered by the one S tile
constexpr int THREADS = 224;
constexpr uint32_t Q_BYTES = BQ * HD * 2;     // 16 KB
constexpr uint32_t KV_BYTES = NK * HD * 2;    // 32 KB each for K and V
constexpr int TAIL_ROWS = 16;                 // the remainder key travels as a 16-row TMA box (rows 1..15: next sequence / zero fill)
constexpr uint32_t TAIL_BYTES = TAIL_ROWS * HD * 2;   // 2 KB each for the remainder key's K tile and V tile
constexpr uint32_t BAR_BYTES = 256;
constexpr uint32_t SMEM_BYTES = 2 * Q_BYTES + 2 * KV_BYTES + 2 * TAIL_BYTES + BAR_BYTES;
static_assert(SMEM_BYTES <= 115712, "two CTAs per SM");
constexpr uint32_t TMEM_COLS = 256;
constexpr uint32_t S_COL = 0, P_COL = 0, O_COL = 128;
constexpr uint32_t T_COL = 192;   // remainder key's scores (N = 16 MMA, column 0 is the key), written after S is consumed

__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(ptx::smem_u32(p)));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(ptx::smem_u32(p)));
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
                 "{%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// tcgen05.wait::ld that names the registers an in-flight tcgen05.ld fills (see attention_tc.cu)
__device__ __forceinline__ void tmem_ld_wait_regs(uint32_t (&v)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                   "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                   "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x1(uint32_t taddr, uint32_t& v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
}
// 32 lanes x 16 columns: registers -> TMEM (thread t writes lane base_lane + t)
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]: the A operand (bf16 pairs, one row per lane, K along the columns) comes from TMEM
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// running maximum of one 32-column chunk of a score row; keys (block-local) >= khi are masked
template <bool FULL>
__device__ __forceinline__ void max_chunk(const uint32_t (&v)[32], int c, int khi, float (&mx)[4]) {
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        const float s = __uint_as_float(v[i]);
        if (FULL) mx[i & 3] = fmaxf(mx[i & 3], s);
        else mx[i & 3] = (c * 32 + i < khi) ? fmaxf(mx[i & 3], s) : mx[i & 3];
    }
}
// p = exp2(s * scale - m) for one 32-key chunk, row sum, bf16 pairs -> TMEM columns P_COL + 16 c .. + 15
template <bool FULL>
__device__ __forceinline__ void exp_chunk(const uint32_t (&v)[32], int c, int khi, float scale_log2e, float m_safe,
                                          float (&ls)[4], uint32_t p_addr) {
    uint32_t pk[16];
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
        const float s0 = __uint_as_float(v[i]), s1 = __uint_as_float(v[i + 1]);
        // (the clamp only matters for a score more than 2^132 above the first-chunk maximum: it keeps P, l and O far inside fp32 range — such a
        // key then simply takes the whole row — instead of producing inf / NaN)
        float p0 = ex2(fminf(fmaf(s0, scale_log2e, -m_safe), 100.0f));
        float p1 = ex2(fminf(fmaf(s1, scale_log2e, -m_safe), 100.0f));
        if (!FULL) {
            p0 = (c * 32 + i < khi) ? p0 : 0.f;
            p1 = (c * 32 + i + 1 < khi) ? p1 : 0.f;
        }
        ls[(i >> 1) & 3] += p0 + p1;
        pk[i >> 1] = pack2(p0, p1);
    }
    tmem_st_32x32b_x16(p_addr + 16 * c, pk);
}

// (Tried and measured slower, 200 vs 176 us per ViT-L-14 layer in one run: letting an elected softmax thread issue P V and the
//  next item's S itself after a 128-thread named barrier, to save the two mbarrier hand-offs through warp 1 — the issuing
//  thread's waits and the divergence they cause inside its warp cost more than the hops.)
template <int MASK>
__global__ void __launch_bounds__(THREADS, 2)
attention_os_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_tail,
                    const __nv_bfloat16* __restrict__ qkv,
                    __nv_bfloat16* __restrict__ out, int S, int W, int H, const int32_t* __restrict__ kv_len,
                    float scale_log2e, int s_main, int has_tail, int total_units) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sQ = smem;                         // two 16 KB tiles
    uint8_t* sK = sQ + 2 * Q_BYTES;             // 256 keys x 64 dims, K-major 128B-swizzled (two TMA boxes)
    uint8_t* sV = sK + KV_BYTES;                // 256 keys x 64 dims: the MN-major B operand of P V
    uint8_t* sKt = sV + KV_BYTES;               // remainder key: K rows s_main .. s_main + 15 (row 0 is the key)
    uint8_t* sVt = sKt + TAIL_BYTES;            // ... and its V rows (row 0 = 128 contiguous bytes: swizzle is the identity there)
    uint64_t* bars = reinterpret_cast<uint64_t*>(sVt + TAIL_BYTES);
    uint64_t* q_full = bars;          // [2]
    uint64_t* q_empty = bars + 2;     // [2]
    uint64_t* k_full = bars + 4;
    uint64_t* k_empty = bars + 5;
    uint64_t* v_full = bars + 6;
    uint64_t* v_empty = bars + 7;
    uint64_t* s_full = bars + 8;
    uint64_t* p_full = bars + 9;
    uint64_t* o_full = bars + 10;
    uint64_t* tmem_free = bars + 11;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);
    const __nv_bfloat16* sTailV = reinterpret_cast<const __nv_bfloat16*>(sVt);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    if ((ptx::smem_u32(smem) & 1023u) != 0) __trap();
    const int q_blocks = 2;   // 129 <= S <= 257: rows 0..127 and 128..255 (a 257th row is warp 6's remainder row)

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmap);
        ptx::prefetch_tmap(&tmap_tail);
        for (int i = 0; i < 2; ++i) {
            ptx::mbar_init(&q_full[i], 1);
            ptx::mbar_init(&q_empty[i], 1);   // the commit after the item's last MMA that reads the Q tile
        }
        ptx::mbar_init(k_full, 1);
        ptx::mbar_init(k_empty, 2);           // the last S MMA's commit + warp 6 (remainder row)
        ptx::mbar_init(v_full, 1);
        ptx::mbar_init(v_empty, has_tail ? 6 : 2);   // the last P V's commit + warp 6 (+ the 4 epilogue warps: remainder V row)
        ptx::mbar_init(s_full, 1);
        ptx::mbar_init(p_full, 4);
        ptx::mbar_init(o_full, 1);
        ptx::mbar_init(tmem_free, 4);
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        ptx::tmem_alloc_n<TMEM_COLS>(tmem_slot);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // The two MMA groups of an item, issued by ONE thread (warp 1's lane 0, or the softmax warps' elected thread).
    auto issue_s = [&](uint32_t n, uint32_t uc, int qb) {
        constexpr uint32_t idesc_s = ptx::make_idesc_f16_major(1, BQ, NK, 0, 0);
        const uint32_t buf = n & 1;
        ptx::mbar_wait(&q_full[buf], (n >> 1) & 1);
        if (qb == 0) ptx::mbar_wait(k_full, uc & 1);
        ptx::tc_fence_after();
        const uint32_t q_base = ptx::smem_u32(sQ + buf * Q_BYTES);
        const uint32_t k_base = ptx::smem_u32(sK);
#pragma unroll
        for (int k = 0; k < HD / 16; ++k)
            ptx::umma_f16(tmem_base + S_COL, ptx::make_desc_k_sw128(q_base + k * 32),
                          ptx::make_desc_k_sw128(k_base + k * 32), idesc_s, k != 0 ? 1u : 0u);
        ptx::umma_commit(s_full);
        if (!has_tail) {
            ptx::umma_commit(&q_empty[buf]);
            if (qb == q_blocks - 1) ptx::umma_commit(k_empty);
        }
    };
    auto issue_pv = [&](uint32_t n, uint32_t uc, int qb) {
        constexpr uint32_t idesc_o = ptx::make_idesc_f16_major(1, BQ, HD, 0, 1);   // A (P) K-major in TMEM, B (V) MN-major
        constexpr uint32_t idesc_t = ptx::make_idesc_f16_major(1, BQ, TAIL_ROWS, 0, 0);   // Q x (remainder key tile)^T
        const uint32_t buf = n & 1;
        if (qb == 0) ptx::mbar_wait(v_full, uc & 1);
        ptx::tc_fence_after();
        const uint32_t v_base = ptx::smem_u32(sV);
#pragma unroll
        for (int k = 0; k < NK / 16; ++k)
            umma_f16_ts(tmem_base + O_COL, tmem_base + P_COL + k * 8,
                        ptx::make_desc_mn_sw128(v_base + k * 16 * 128, 8192, 1024), idesc_o, k != 0 ? 1u : 0u);
        if (has_tail) {
            // the remainder key's scores for the item's 128 rows: a 16-column MMA into columns that S no longer needs
            // (all of S has been consumed once P is complete); the epilogue reads column T_COL
            const uint32_t q_base = ptx::smem_u32(sQ + buf * Q_BYTES);
            const uint32_t kt_base = ptx::smem_u32(sKt);
#pragma unroll
            for (int k = 0; k < HD / 16; ++k)
                ptx::umma_f16(tmem_base + T_COL, ptx::make_desc_k_sw128(q_base + k * 32),
                              ptx::make_desc_k_sw128(kt_base + k * 32), idesc_t, k != 0 ? 1u : 0u);
            ptx::umma_commit(&q_empty[buf]);
            if (qb == q_blocks - 1) ptx::umma_commit(k_empty);
        }
        ptx::umma_commit(o_full);
        if (qb == q_blocks - 1) ptx::umma_commit(v_empty);
    };

    // every role walks units u = blockIdx.x, + gridDim.x, ... (unit = (batch, head)) and the unit's two query blocks;
    // n = items (query blocks) done so far, uc = units done so far.  Unit u is (batch, head) ur = total_units - 1 - u:
    // the QKV GEMM wrote the packed qkv matrix in ascending row order, so its last rows are the ones still in L2.
    if (warp == 0) {
        // ================================================================== TMA producer
        if (lane == 0) {
            uint32_t n = 0, uc = 0;
            for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++uc) {
                const int ur = total_units - 1 - u;
                const int b = ur / H, h = ur - b * H;
                const int row_base = b * S;
                for (int qb = 0; qb < q_blocks; ++qb, ++n) {
                    const uint32_t buf = n & 1;
                    ptx::mbar_wait(&q_empty[buf], ((n >> 1) & 1) ^ 1);
                    ptx::mbar_arrive_expect_tx(&q_full[buf], Q_BYTES);
                    ptx::tma_load_2d(sQ + buf * Q_BYTES, &tmap, &q_full[buf], h * HD, row_base + qb * BQ, ptx::kEvictNormal);
                    if (qb == 0) {
                        ptx::mbar_wait(k_empty, (uc & 1) ^ 1);
                        ptx::mbar_arrive_expect_tx(k_full, KV_BYTES + (has_tail ? TAIL_BYTES : 0));
                        ptx::tma_load_2d(sK, &tmap, k_full, W + h * HD, row_base, ptx::kEvictNormal);
                        ptx::tma_load_2d(sK + KV_BYTES / 2, &tmap, k_full, W + h * HD, row_base + 128, ptx::kEvictNormal);
                        if (has_tail)
                            ptx::tma_load_2d(sKt, &tmap_tail, k_full, W + h * HD, row_base + s_main, ptx::kEvictNormal);
                    } else {
                        ptx::mbar_wait(v_empty, (uc & 1) ^ 1);
                        ptx::mbar_arrive_expect_tx(v_full, KV_BYTES + (has_tail ? TAIL_BYTES : 0));
                        ptx::tma_load_2d(sV, &tmap, v_full, 2 * W + h * HD, row_base, ptx::kEvictNormal);
                        ptx::tma_load_2d(sV + KV_BYTES / 2, &tmap, v_full, 2 * W + h * HD, row_base + 128,
                                         ptx::kEvictNormal);
                        if (has_tail)
                            ptx::tma_load_2d(sVt, &tmap_tail, v_full, 2 * W + h * HD, row_base + s_main, ptx::kEvictNormal);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================================================================== MMA issuer
        uint32_t n = 0, uc = 0;
        for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++uc) {
            for (int qb = 0; qb < q_blocks; ++qb, ++n) {
                if (n > 0) ptx::mbar_wait(tmem_free, (n - 1) & 1);   // the previous item's O has been read out
                if (lane == 0) issue_s(n, uc, qb);
                __syncwarp();
                ptx::mbar_wait(p_full, n & 1);       // P of this item is in TMEM (and S fully consumed)
                if (lane == 0) issue_pv(n, uc, qb);
                __syncwarp();
            }
        }
    } else if (warp == 6) {
        // ================================================================== remainder key + remainder query row
        uint32_t uc = 0;
        const size_t ld = (size_t)3 * W;
        const int gq = lane >> 2, tq = lane & 3;
        for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++uc) {
            const int ur = total_units - 1 - u;
            const int b = ur / H, h = ur - b * H;
            const int row_base = b * S;
            int len = S;
            if (MASK == MASK_KEYLEN) len = min(S, max(kv_len[b], 0));
            {
                // (the remainder KEY is the tensor core's job: a 16-row K tile + a 16-column MMA per item, see the MMA warp)
                const int nu = u + gridDim.x;
                if (has_tail && lane == 0 && nu < total_units) {   // the next unit's remainder row: into L2 ahead of time
                    const int nur = total_units - 1 - nu;
                    const int nb = nur / H, nh = nur - nb * H;
                    const __nv_bfloat16* nrow = qkv + ((size_t)nb * S + s_main) * ld + nh * HD;
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(nrow));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(nrow + W));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(nrow + 2 * W));
                }
                // K / V work of this warp happens as soon as the unit's tiles have landed: the sooner this warp hands
                // K / V back, the sooner the producer can start the next unit's loads (they are single buffered)
                ptx::mbar_wait(k_full, uc & 1);
                ptx::mbar_wait(v_full, uc & 1);
                // ---- remainder row (query index s_main) against the 256 keys in shared memory, row 0 of 16-row mma tiles
                if (has_tail && s_main < S) {
                    const int trow = s_main;
                    const int tlimit = len;
                    uint32_t qf[4][4];
                    float o[8][4];
                    float row_max = -INFINITY, row_sum = 0.f;
                    const __nv_bfloat16* qrow_p = qkv + ((size_t)row_base + trow) * ld + h * HD;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        qf[ks][0] = gq == 0 ? *reinterpret_cast<const uint32_t*>(qrow_p + ks * 16 + 2 * tq) : 0u;
                        qf[ks][1] = 0u;
                        qf[ks][2] = gq == 0 ? *reinterpret_cast<const uint32_t*>(qrow_p + ks * 16 + 8 + 2 * tq) : 0u;
                        qf[ks][3] = 0u;
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i)
#pragma unroll
                        for (int e = 0; e < 4; ++e) o[i][e] = 0.f;
                    const __nv_bfloat16* kt0 = reinterpret_cast<const __nv_bfloat16*>(sK);
                    const __nv_bfloat16* vt0 = reinterpret_cast<const __nv_bfloat16*>(sV);
                    const int mat = lane >> 3, rr8 = lane & 7;
                    auto tile_at = [](const __nv_bfloat16* tile, int row, int chunk) {
                        return tile + row * HD + ((chunk ^ (row & 7)) << 3);
                    };
#pragma unroll 1
                    for (int j = 0; j < 2; ++j) {
                        const __nv_bfloat16* kt = kt0 + j * 128 * HD;
                        const __nv_bfloat16* vt = vt0 + j * 128 * HD;
                        float sc[16][4];
#pragma unroll
                        for (int i = 0; i < 16; ++i)
#pragma unroll
                            for (int e = 0; e < 4; ++e) sc[i][e] = 0.f;
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
                            for (int np = 0; np < 8; ++np) {
                                uint32_t kf[4];
                                ldmatrix_x4(kf, tile_at(kt, np * 16 + (mat >> 1) * 8 + rr8, ks * 2 + (mat & 1)));
                                mma_bf16(sc[2 * np], qf[ks], kf[0], kf[1]);
                                mma_bf16(sc[2 * np + 1], qf[ks], kf[2], kf[3]);
                            }
                        }
                        float mx = row_max;
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const int key = j * 128 + i * 8 + 2 * tq + e;
                                const float v = (key < tlimit && key < s_main) ? sc[i][e] * scale_log2e : -INFINITY;
                                sc[i][e] = v;
                                mx = fmaxf(mx, v);
                            }
                        }
                        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
                        const float msafe = mx == -INFINITY ? 0.f : mx;
                        const float corr = ex2(row_max - msafe);
                        row_max = mx;
                        row_sum *= corr;
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            o[i][0] *= corr;
                            o[i][1] *= corr;
                        }
                        float ps = 0.f;
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const float pv = ex2(sc[i][e] - msafe);
                                ps += pv;
                                sc[i][e] = pv;
                            }
                        }
                        row_sum += ps;
#pragma unroll
                        for (int ks = 0; ks < 8; ++ks) {
                            uint32_t pa[4];
                            pa[0] = pack2(sc[2 * ks][0], sc[2 * ks][1]);
                            pa[1] = 0u;
                            pa[2] = pack2(sc[2 * ks + 1][0], sc[2 * ks + 1][1]);
                            pa[3] = 0u;
#pragma unroll
                            for (int dp = 0; dp < 4; ++dp) {
                                uint32_t vf[4];
                                ldmatrix_x4_trans(vf, tile_at(vt, ks * 16 + (mat & 1) * 8 + rr8, dp * 2 + (mat >> 1)));
                                mma_bf16(o[2 * dp], pa, vf[0], vf[1]);
                                mma_bf16(o[2 * dp + 1], pa, vf[2], vf[3]);
                            }
                        }
                    }
                    __syncwarp();
                    if (lane == 0) {   // K / V of this unit are no longer needed by this warp
                        ptx::mbar_arrive(k_empty);
                        ptx::mbar_arrive(v_empty);
                    }
                    if (s_main < tlimit) {   // the remainder key against the remainder row
                        const __nv_bfloat16* krow = qkv + ((size_t)row_base + s_main) * ld + W + h * HD;
                        const float2 qpair = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(qrow_p)[lane]);
                        const float2 kf2 = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(krow)[lane]);
                        float sd = qpair.x * kf2.x + qpair.y * kf2.y;
#pragma unroll
                        for (int off = 16; off > 0; off >>= 1) sd += __shfl_xor_sync(0xffffffffu, sd, off);
                        const float scv = sd * scale_log2e;
                        const float m_new = fmaxf(row_max, scv);
                        const float alpha = ex2(row_max - m_new);
                        const float pe = ex2(scv - m_new);
                        const float pbv = __bfloat162float(__float2bfloat16_rn(pe));
                        row_sum = row_sum * alpha + (tq == 0 ? pe : 0.f);
                        row_max = m_new;
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float2 vf2 = __bfloat1622float2(
                                *reinterpret_cast<const __nv_bfloat162*>(krow + W + i * 8 + 2 * tq));
                            o[i][0] = fmaf(o[i][0], alpha, pbv * vf2.x);
                            o[i][1] = fmaf(o[i][1], alpha, pbv * vf2.y);
                        }
                    }
                    row_sum += __shfl_xor_sync(0xffffffffu, row_sum, 1);
                    row_sum += __shfl_xor_sync(0xffffffffu, row_sum, 2);
                    const float inv_t = row_sum > 0.f ? 1.f / row_sum : 0.f;
                    if (gq == 0) {
                        __nv_bfloat16* orow = out + ((size_t)row_base + trow) * W + h * HD;
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            *reinterpret_cast<uint32_t*>(orow + i * 8 + 2 * tq) = pack2(o[i][0] * inv_t, o[i][1] * inv_t);
                    }
                } else {
                    __syncwarp();
                    if (lane == 0) {
                        ptx::mbar_arrive(k_empty);
                        ptx::mbar_arrive(v_empty);
                    }
                }
            }
        }
    } else {
        // ================================================================== softmax / epilogue: thread == query row
        const int sp = warp & 3;
        const int r = sp * 32 + lane;
        const uint32_t lane_addr = tmem_base + (uint32_t(sp * 32) << 16);
        uint32_t n = 0;
        for (int u = blockIdx.x; u < total_units; u += gridDim.x) {
            const int ur = total_units - 1 - u;
            const int b = ur / H, h = ur - b * H;
            const int row_base = b * S;
            int len = S;
            if (MASK == MASK_KEYLEN) len = min(S, max(kv_len[b], 0));
            const int khi = min(len, s_main);            // keys >= khi of the S tile are masked
            const bool full = khi >= NK;
            const bool has_tail_key = has_tail && s_main < len;
            for (int qb = 0; qb < q_blocks; ++qb, ++n) {
                const int qrow = qb * BQ + r;
                const bool row_valid = qrow < min(S, s_main);
                ptx::mbar_wait(s_full, n & 1);
                ptx::tc_fence_after();
                uint32_t va[32], vb[32];
                // ---- ONE pass over S.  softmax(s) = exp2(s' - ref) / sum exp2(s' - ref) for ANY reference, so the
                // exponent reference does not have to be the row maximum — only close enough that nothing overflows:
                // ref = (maximum of the row's first 32 scores) + 32.  A later score may exceed that maximum by up to
                // 2^132 before the clamp in exp_chunk engages (l and O stay far inside fp32 range), scores more than 2^94 below it flush to zero next to a term >= 2^-32, and
                // P, l and O are floating point (bf16 / fp32: 8 exponent bits), so the common factor 2^-32 costs no
                // precision; it cancels in O / l.  (attention_tc.cu needs the running maximum because it accumulates
                // over key blocks; here all 256 keys are in TMEM at once.)
                ptx::tmem_ld_32x32b_x32(lane_addr + S_COL, va);
                tmem_ld_wait_regs(va);
                ptx::tmem_ld_32x32b_x32(lane_addr + S_COL + 32, vb);
                float c0[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
                if (full) max_chunk<true>(va, 0, khi, c0);
                else max_chunk<false>(va, 0, khi, c0);
                const float cmax = fmaxf(fmaxf(c0[0], c0[1]), fmaxf(c0[2], c0[3]));
                const float m_run0 = cmax == -INFINITY ? -INFINITY : fmaf(cmax, scale_log2e, 32.0f);
                const float m_safe = m_run0 == -INFINITY ? 0.f : m_run0;
                float ls4[4] = {0.f, 0.f, 0.f, 0.f};
                const uint32_t p_addr = lane_addr + P_COL;
#pragma unroll 1
                for (int c = 0; c < NK / 32; c += 2) {
                    if (c > 0) {
                        tmem_ld_wait_regs(va);
                        ptx::tmem_ld_32x32b_x32(lane_addr + S_COL + (c + 1) * 32, vb);
                    }
                    if (full) exp_chunk<true>(va, c, khi, scale_log2e, m_safe, ls4, p_addr);
                    else exp_chunk<false>(va, c, khi, scale_log2e, m_safe, ls4, p_addr);
                    tmem_ld_wait_regs(vb);
                    if (c + 2 < NK / 32) ptx::tmem_ld_32x32b_x32(lane_addr + S_COL + (c + 2) * 32, va);
                    if (full) exp_chunk<true>(vb, c + 1, khi, scale_log2e, m_safe, ls4, p_addr);
                    else exp_chunk<false>(vb, c + 1, khi, scale_log2e, m_safe, ls4, p_addr);
                }
                float l_run = (ls4[0] + ls4[1]) + (ls4[2] + ls4[3]);
                float m_run = m_run0;
                ptx::tmem_st_wait();
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(p_full);
                ptx::mbar_wait(o_full, n & 1);
                ptx::tc_fence_after();
                ptx::tmem_ld_32x32b_x32(lane_addr + O_COL, va);
                ptx::tmem_ld_32x32b_x32(lane_addr + O_COL + 32, vb);
                uint32_t tsc = 0;
                if (has_tail) tmem_ld_32x32b_x1(lane_addr + T_COL, tsc);   // q_row . remainder key (fp32 accumulator)
                ptx::tmem_ld_wait();
                // O is in registers: the next item's S may overwrite the accumulator columns
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(tmem_free);
                // ---- remainder key: online update of (m, l); folded into the output below
                float t_alpha = 1.f, t_p = 0.f;
                if (has_tail_key) {
                    const float sc = __uint_as_float(tsc) * scale_log2e;
                    const float m_new = fmaxf(m_run, sc);
                    t_alpha = ex2(m_run - m_new);
                    const float pe = ex2(sc - m_new);
                    t_p = __bfloat162float(__float2bfloat16_rn(pe));   // the tensor-core path rounds P to bf16 too
                    l_run = l_run * t_alpha + pe;
                    m_run = m_new;
                }
                const float inv = l_run > 0.f ? 1.f / l_run : 0.f;
                if (row_valid) {
                    uint4* d4 = reinterpret_cast<uint4*>(out + ((size_t)row_base + qrow) * W + h * HD);
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf) {
                        const uint32_t* vv = hf == 0 ? va : vb;
                        float o[32];
#pragma unroll
                        for (int i = 0; i < 32; ++i) o[i] = __uint_as_float(vv[i]);
                        if (has_tail_key) {
                            const uint4* vp = reinterpret_cast<const uint4*>(sTailV) + hf * 4;
#pragma unroll
                            for (int x = 0; x < 4; ++x) {
                                const uint4 v4 = vp[x];
                                const uint32_t ve[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    const float2 f2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ve[e]));
                                    o[8 * x + 2 * e] = fmaf(o[8 * x + 2 * e], t_alpha, t_p * f2.x);
                                    o[8 * x + 2 * e + 1] = fmaf(o[8 * x + 2 * e + 1], t_alpha, t_p * f2.y);
                                }
                            }
                        }
#pragma unroll
                        for (int x = 0; x < 4; ++x)
                            d4[hf * 4 + x] = make_uint4(pack2(o[8 * x] * inv, o[8 * x + 1] * inv),
                                                        pack2(o[8 * x + 2] * inv, o[8 * x + 3] * inv),
                                                        pack2(o[8 * x + 4] * inv, o[8 * x + 5] * inv),
                                                        pack2(o[8 * x + 6] * inv, o[8 * x + 7] * inv));
                    }
                }
                if (has_tail && qb == q_blocks - 1) {
                    // the remainder key's V row (sVt) has been read for the unit's last item: the V buffers may be refilled
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(v_empty);
                }
            }
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

}  // namespace os

bool os_supported(int S, int mask) {
    return S > os::BQ && S <= os::NK + 1 && (mask == MASK_NONE || mask == MASK_KEYLEN);
}

int launch_os(const __nv_bfloat16* qkv, __nv_bfloat16* out, int B, int S, int W, int H, int mask, const int32_t* kv_len,
              cudaStream_t stream) {
    if (B <= 0) return 0;
    if (W != H * os::HD) fail(B200_ERR_UNSUPPORTED, "attention: head_dim must be 64 (width %d, heads %d)", W, H);
    if (!os_supported(S, mask)) fail(B200_ERR_INTERNAL, "attention: one-shot kernel does not cover S = %d, mask %d", S, mask);
    if (mask == MASK_KEYLEN && !kv_len) fail(B200_ERR_INTERNAL, "attention: kv_len required for key-length masking");
    static std::once_flag once;
    std::call_once(once, [] {
        const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
        MB_CUDA(cudaFuncSetAttribute(os::attention_os_kernel<MASK_NONE>, attr, (int)os::SMEM_BYTES));
        MB_CUDA(cudaFuncSetAttribute(os::attention_os_kernel<MASK_KEYLEN>, attr, (int)os::SMEM_BYTES));
    });
    CUtensorMap tmap = make_tmap_2d(qkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)3 * W, (uint64_t)B * S,
                                    (uint64_t)3 * W * 2, os::HD, os::BQ, CU_TENSOR_MAP_SWIZZLE_128B);
    // the remainder key (row 256 of a 257-token sequence) of K and of V: 16-row boxes of the same matrix
    CUtensorMap tmap_tail = make_tmap_2d(qkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)3 * W, (uint64_t)B * S,
                                         (uint64_t)3 * W * 2, os::HD, os::TAIL_ROWS, CU_TENSOR_MAP_SWIZZLE_128B);
    const float scale_log2e = 0.125f * 1.4426950408889634f;
    int device = 0;
    MB_CUDA(cudaGetDevice(&device));
    const bool tail = S == os::NK + 1;
    const int s_main = tail ? os::NK : S;
    const int total_units = B * H;
    const int grid = std::min(2 * sm_count(device), total_units);
    if (mask == MASK_NONE)
        os::attention_os_kernel<MASK_NONE><<<grid, os::THREADS, os::SMEM_BYTES, stream>>>(
            tmap, tmap_tail, qkv, out, S, W, H, kv_len, scale_log2e, s_main, tail ? 1 : 0, total_units);
    else
        os::attention_os_kernel<MASK_KEYLEN><<<grid, os::THREADS, os::SMEM_BYTES, stream>>>(
            tmap, tmap_tail, qkv, out, S, W, H, kv_len, scale_log2e, s_main, tail ? 1 : 0, total_units);
    MB_CUDA(cudaGetLastError());
    return 1;
}

}  // namespace attention
}  // namespace mb
