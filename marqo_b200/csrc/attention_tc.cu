// tcgen05 flash attention (head_dim 64, S <= a few thousand, bf16 in / fp32 softmax / bf16 out).
//
// PERSISTENT: 2 CTAs per SM loop over work items (batch, head, 128-query block); barriers, TMEM and the tensor map are
// set up once per CTA and the producer / MMA warps run ahead into the next item while the softmax warps finish the
// current one (per-CTA launch + set-up + first-load latency used to cost ~3 us per 128-query block — more than the
// two key blocks of a 257-token ViT sequence themselves).
// Warp 0: TMA producer (Q per item, K/V blocks of 128 keys through a 2-stage ring, all 128B-swizzled straight from the
// packed qkv matrix).  Warp 1: single-thread tcgen05.mma issuer:
//   S = Q K_j^T   (M=128, N=128, K=64;  A, B K-major)          -> TMEM columns [0,128)
//   O += P_j V_j  (M=128, N=64,  K=128; A = P K-major from smem, B = V MN-major as loaded)  -> TMEM columns [128,192)
// Warps 2-5: softmax, ONE THREAD PER QUERY ROW (TMEM lane == row): one pass over the row's 128 scores in TMEM against a
// lazy exponent reference (exp2 / sum / bf16 P written to smem in the UMMA K-major swizzled layout, the exact maximum
// tracked on the side; a warp whose reference falls too far behind redoes the block exactly), rescale of the O
// accumulator through tcgen05.ld/st when the reference moves, final 1/l scaling and the bf16 store.  S of block g + 1 is issued before P.V of
// block g (also across items), so the next scores are ready when the softmax warps come back.
// Warp 6: the remainder key and query row of a sequence such as 257 = 2 * 128 + 1 (ViT class token): the key's scores
// against the 128 rows of the item and its V row are staged in smem for the epilogue; the row runs on mma.sync
// against the K / V tiles while they sit in shared memory.
// 113 KB smem + 256 TMEM columns per CTA -> two CTAs per SM, so one CTA's softmax overlaps the other's MMAs.
// BIAS (MPNet): a learned relative-position bias per (head, key - query) enters every score before the softmax; warp 6
// stages the item's head row of the bias in shared memory instead of handling a remainder key / row.
#include <algorithm>
#include <mutex>

#include "attention.cuh"
#include "ptx.cuh"

namespace mb {
namespace attention {

namespace tc {

constexpr int HD = 64;
constexpr int BQ = 128;
constexpr int BKV = 128;
constexpr int THREADS = 224;   // warp 0 TMA, warp 1 MMA, warps 2-5 softmax, warp 6 remainder rows
constexpr int KV_STAGES = 2;
constexpr uint32_t Q_BYTES = BQ * HD * 2;        // 16 KB
constexpr uint32_t KV_TILE_BYTES = BKV * HD * 2;  // 16 KB each for K and V
constexpr uint32_t P_BYTES = BQ * BKV * 2;        // 32 KB (two 64-key K-major chunks)
constexpr uint32_t TAILS_BYTES = BQ * 4;                     // the remainder key's score for each of the 128 rows
constexpr uint32_t TAILV_BYTES = HD * 2;                     // the remainder key's V row
// 115712 B: two CTAs (+ 1 KB of system-reserved smem each) fill the SM's 228 KB exactly
constexpr uint32_t SMEM_BYTES =
    Q_BYTES + KV_STAGES * 2 * KV_TILE_BYTES + P_BYTES + 128 + TAILS_BYTES + TAILV_BYTES;
static_assert(SMEM_BYTES <= 115712, "two CTAs per SM");
// BIAS: the staged head row of the relative-position bias (REL_T fp32) takes the place of the remainder key's scores
// and V row: there is no room for both, so sequences of k * 128 + 1 tokens run their last key / query on a masked block
constexpr uint32_t BIAS_ROW_BYTES = (REL_T * 4 + 15) / 16 * 16;
constexpr uint32_t SMEM_BYTES_BIAS = Q_BYTES + KV_STAGES * 2 * KV_TILE_BYTES + P_BYTES + 128 + BIAS_ROW_BYTES;
static_assert(SMEM_BYTES_BIAS <= 115712, "two CTAs per SM");
constexpr uint32_t TMEM_COLS = 256;
constexpr uint32_t S_COL = 0, O_COL = 128;

__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
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
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

// tcgen05.wait::ld that names the registers an in-flight tcgen05.ld fills: every use of v[] after this statement depends
// on it, so the compiler cannot schedule arithmetic on a prefetched chunk ahead of the wait.
__device__ __forceinline__ void tmem_ld_wait_regs(uint32_t (&v)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                   "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                   "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :
                 : "memory");
}

// Relative-position bias of key - query = d (log2 units): sB points at the staged head row's d = 0 entry.
__device__ __forceinline__ float rel_bias(const float* sB, int d) { return sB[min(max(d, -REL_D), REL_D)]; }

// One 32-key chunk of a score row: p = exp2(s * scale - m_safe) for the keys in [klo, khi) (block-local indices), 0 for
// the others; running raw maximum, row sum, bf16 P into the K-major 128B-swizzled A-operand layout.
// BIAS: the scores are x = s * scale_log2e + bias (dk = block key 0 - query) and mx tracks x, not the raw s.
template <bool FULL, bool BIAS = false>
__device__ __forceinline__ void softmax_chunk(const uint32_t (&v)[32], int c, int klo, int khi, float scale_log2e,
                                              float m_safe, float& lsum, float& mx, uint8_t* sP, int r,
                                              const float* sB = nullptr, int dk = 0) {
    uint32_t pk[16];
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
        const float s0 = __uint_as_float(v[i]), s1 = __uint_as_float(v[i + 1]);
        float p0, p1;
        if constexpr (BIAS) {
            const int k0 = c * 32 + i;
            const float x0 = fmaf(s0, scale_log2e, rel_bias(sB, dk + k0));
            const float x1 = fmaf(s1, scale_log2e, rel_bias(sB, dk + k0 + 1));
            const bool ok0 = FULL || (k0 >= klo && k0 < khi), ok1 = FULL || (k0 + 1 >= klo && k0 + 1 < khi);
            mx = ok0 ? fmaxf(mx, x0) : mx;
            mx = ok1 ? fmaxf(mx, x1) : mx;
            p0 = ok0 ? ex2(x0 - m_safe) : 0.f;
            p1 = ok1 ? ex2(x1 - m_safe) : 0.f;
        } else if (FULL) {
            mx = fmaxf(mx, fmaxf(s0, s1));
            p0 = ex2(fmaf(s0, scale_log2e, -m_safe));
            p1 = ex2(fmaf(s1, scale_log2e, -m_safe));
        } else {
            const int k0 = c * 32 + i;
            const bool ok0 = k0 >= klo && k0 < khi, ok1 = k0 + 1 >= klo && k0 + 1 < khi;
            mx = ok0 ? fmaxf(mx, s0) : mx;
            mx = ok1 ? fmaxf(mx, s1) : mx;
            p0 = ok0 ? ex2(fmaf(s0, scale_log2e, -m_safe)) : 0.f;
            p1 = ok1 ? ex2(fmaf(s1, scale_log2e, -m_safe)) : 0.f;
        }
        lsum += p0 + p1;
        pk[i >> 1] = pack2(p0, p1);
    }
    // keys c*32 .. c*32+31 -> chunk (c >> 1), 16-byte units (c & 1) * 4 .. +3 of row r
    uint8_t* rowp = sP + (size_t)(c >> 1) * (BQ * 128) + (size_t)r * 128;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int unit = (c & 1) * 4 + u;
        *reinterpret_cast<uint4*>(rowp + ((unit ^ (r & 7)) << 4)) =
            make_uint4(pk[4 * u], pk[4 * u + 1], pk[4 * u + 2], pk[4 * u + 3]);
    }
}

// work item -> (batch, head, query block); consecutive items share (batch, head) so the two CTAs that process them
// at the same time read K / V once from HBM and once from L2
struct Item {
    int b, h, q0, qb;
};
__device__ __forceinline__ Item decode_item(int it, int q_blocks, int H) {
    Item w;
    w.qb = it % q_blocks;
    const int bh = it / q_blocks;
    w.h = bh % H;
    w.b = bh / H;
    w.q0 = w.qb * BQ;
    return w;
}

// PACKED (S < 128): an item is a GROUP of pack = 128 / S consecutive sequences sharing one 128-row tile; w.b is the
// group index, the tile's valid rows / keys are the group's nseq * S tokens and the mask is block-diagonal (a row only
// sees the keys of its own sequence) — see the softmax warps.
template <int MASK, bool PACKED>
__device__ __forceinline__ void item_extent(const Item& w, int S, int s_main, const int32_t* kv_len, int& len, int& kend,
                                            int& nkb, int pack = 1, int B = 0) {
    if (PACKED) {
        const int nseq = max(0, min(pack, B - w.b * pack));
        len = kend = nseq * S;
        nkb = nseq > 0 ? 1 : 0;
        return;
    }
    len = S;
    if (MASK == MASK_KEYLEN) len = min(S, max(kv_len[w.b], 0));
    kend = min(len, s_main);
    if (MASK == MASK_CAUSAL) kend = min(kend, w.q0 + BQ);
    nkb = (kend + BKV - 1) / BKV;
}

// Two CTAs per SM: 14 warps over 4 schedulers put 4 warps on one of them, and a scheduler's register partition
// (16384 registers) holds 4 warps only up to 128 registers each — a 144-register build (tried in round 2) silently
// dropped to ONE CTA per SM and ran 1.85x slower.
// BIAS: every score gets the relative-position bias of its head and of key - query (positions within the sequence, also
// in packed tiles) before the softmax; warp 6 stages the item's head row of bias_log2 [H, REL_T] in shared memory
// instead of handling a remainder key / row (the launcher never passes one).
template <int MASK, bool PACKED, bool BIAS>
__global__ void __launch_bounds__(THREADS, 2)
attention_tc_kernel(const __grid_constant__ CUtensorMap tmap, const __nv_bfloat16* __restrict__ qkv,
                    __nv_bfloat16* __restrict__ out, int S, int W, int H, const int32_t* __restrict__ kv_len,
                    float scale_log2e, int s_main, int inline_tail_rows, int q_blocks, int total_items, int pack, int B,
                    const float* __restrict__ bias_log2) {
    const int stride = PACKED ? pack * S : S;   // rows between the bases of consecutive sequences / groups
    // Keys [0, s_main) go through the tensor cores in blocks of 128; the few keys [s_main, S) of a sequence length
    // such as 257 = 2 * 128 + 1 (ViT class token) are folded in on the CUDA cores in the epilogue instead of paying
    // for a whole extra 128-wide block.
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sQ = smem;
    uint8_t* sKV = sQ + Q_BYTES;                       // stage s: K at sKV + s*32K, V at +16K
    uint8_t* sP = sKV + KV_STAGES * 2 * KV_TILE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sP + P_BYTES);
    uint64_t* q_full = bars;
    uint64_t* kv_full = bars + 1;    // [2]
    uint64_t* kv_empty = bars + 3;   // [2]
    uint64_t* s_full = bars + 5;
    uint64_t* s_free = bars + 6;
    uint64_t* p_full = bars + 7;
    uint64_t* pv_done = bars + 8;
    uint64_t* q_empty = bars + 9;
    uint64_t* tail_full = bars + 10;    // the remainder key's scores + V row are staged (warp 6 -> softmax warps)
    uint64_t* tail_empty = bars + 11;   // ... and have been consumed (BIAS: the same for the bias row)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);
    float* sTailS = reinterpret_cast<float*>(sP + P_BYTES + 128);
    __nv_bfloat16* sTailV = reinterpret_cast<__nv_bfloat16*>(sP + P_BYTES + 128 + TAILS_BYTES);
    float* sBias = reinterpret_cast<float*>(sP + P_BYTES + 128);   // BIAS only: bias_log2[h][0 .. REL_T)

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    if ((ptx::smem_u32(smem) & 1023u) != 0) __trap();  // the swizzled tiles need 1024-byte alignment

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmap);
        ptx::mbar_init(q_full, 1);
        // the MMA warp's commit after the item's last S + warp 6 (remainder-key scores; BIAS: warp 6 reads no tile)
        ptx::mbar_init(q_empty, BIAS ? 1 : 2);
        ptx::mbar_init(tail_full, 1);
        ptx::mbar_init(tail_empty, 4);
        for (int i = 0; i < KV_STAGES; ++i) {
            ptx::mbar_init(&kv_full[i], 1);
            ptx::mbar_init(&kv_empty[i], BIAS ? 1 : 2);   // the MMA warp's commit + the remainder-row warp
        }
        ptx::mbar_init(s_full, 1);
        ptx::mbar_init(s_free, 4);
        ptx::mbar_init(p_full, 4);
        ptx::mbar_init(pv_done, 1);
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

    // Every role walks the same item sequence and keeps its own running counters: n = items done, g = key blocks done
    // (ring stage g & 1, ring phase (g >> 1) & 1; the per-block barriers flip with g & 1, the per-item ones with n & 1).
    if (warp == 0) {
        // ================================================================== TMA producer
        if (lane == 0) {
            uint32_t n = 0, g = 0;
            for (int it = blockIdx.x; it < total_items; it += gridDim.x, ++n) {
                const Item w = decode_item(it, q_blocks, H);
                int len, kend, nkb;
                item_extent<MASK, PACKED>(w, S, s_main, kv_len, len, kend, nkb, pack, B);
                const int row_base = w.b * stride;
                if (n > 0) ptx::mbar_wait(q_empty, (n - 1) & 1);   // the previous item's last S MMA has read Q
                ptx::mbar_arrive_expect_tx(q_full, Q_BYTES);
                ptx::tma_load_2d(sQ, &tmap, q_full, w.h * HD, row_base + w.q0, ptx::kEvictNormal);
                for (int j = 0; j < nkb; ++j, ++g) {
                    const int st = g & 1;
                    ptx::mbar_wait(&kv_empty[st], ((g >> 1) & 1) ^ 1);
                    ptx::mbar_arrive_expect_tx(&kv_full[st], 2 * KV_TILE_BYTES);
                    uint8_t* dst = sKV + (size_t)st * 2 * KV_TILE_BYTES;
                    ptx::tma_load_2d(dst, &tmap, &kv_full[st], W + w.h * HD, row_base + j * BKV, ptx::kEvictLast);
                    ptx::tma_load_2d(dst + KV_TILE_BYTES, &tmap, &kv_full[st], 2 * W + w.h * HD, row_base + j * BKV,
                                     ptx::kEvictLast);
                }
            }
        }
    } else if (warp == 1) {
        // ================================================================== MMA issuer
        // Two cursors walk the same (item, key block) sequence: S of block g + 1 is issued BEFORE P.V of block g, so
        // the tensor core computes the next scores while the softmax warps are still rescaling O and storing P — and,
        // at an item boundary, while they run the epilogue.
        constexpr uint32_t idesc_s = ptx::make_idesc_f16_major(1, BQ, BKV, 0, 0);
        constexpr uint32_t idesc_o = ptx::make_idesc_f16_major(1, BQ, HD, 0, 1);  // B (= V) is MN-major
        struct Cursor {
            int it, j, nkb;
            uint32_t n;
        };
        // skip to the first item (from c.it on) that has key blocks; items without any only hand Q back
        auto settle = [&](Cursor& c, bool owns_q) {
            while (c.it < total_items) {
                const Item w = decode_item(c.it, q_blocks, H);
                int len, kend;
                item_extent<MASK, PACKED>(w, S, s_main, kv_len, len, kend, c.nkb, pack, B);
                if (c.nkb > 0) return;
                if (owns_q) {
                    ptx::mbar_wait(q_full, c.n & 1);
                    if (lane == 0) ptx::mbar_arrive(q_empty);   // nothing to multiply: release Q right away
                    __syncwarp();
                }
                c.it += gridDim.x;
                ++c.n;
            }
        };
        auto advance = [&](Cursor& c, bool owns_q) {
            if (++c.j == c.nkb) {
                c.j = 0;
                c.it += gridDim.x;
                ++c.n;
                settle(c, owns_q);
            }
        };
        Cursor cs{(int)blockIdx.x, 0, 0, 0u}, cp{(int)blockIdx.x, 0, 0, 0u};
        settle(cs, true);
        settle(cp, false);
        uint32_t gs = 0, gp = 0;   // key blocks whose S / P.V have been issued
        auto issue_s = [&]() {
            if (cs.j == 0) ptx::mbar_wait(q_full, cs.n & 1);
            const int st = gs & 1;
            ptx::mbar_wait(&kv_full[st], (gs >> 1) & 1);
            if (gs > 0) ptx::mbar_wait(s_free, (gs - 1) & 1);  // softmax has finished reading S of the previous block
            ptx::tc_fence_after();
            if (lane == 0) {
                const uint32_t q_base = ptx::smem_u32(sQ);
                const uint32_t k_base = ptx::smem_u32(sKV + (size_t)st * 2 * KV_TILE_BYTES);
#pragma unroll
                for (int k = 0; k < HD / 16; ++k)
                    ptx::umma_f16(tmem_base + S_COL, ptx::make_desc_k_sw128(q_base + k * 32),
                                  ptx::make_desc_k_sw128(k_base + k * 32), idesc_s, k != 0 ? 1u : 0u);
                ptx::umma_commit(s_full);
                if (cs.j == cs.nkb - 1) ptx::umma_commit(q_empty);   // Q may be overwritten once these MMAs are done
            }
            __syncwarp();
            ++gs;
            advance(cs, true);
        };
        if (cs.it < total_items) issue_s();
        while (cp.it < total_items) {
            // S of the NEXT block first: the tensor core computes it while the softmax warps are still busy with this
            // block's P, so they go straight from P_g to S_{g+1} and need P.V_g only one pass later — also across an
            // item boundary (252 vs 288 us per ViT-L layer).  Only single-block items (S = 128) prefer their P.V first:
            // there every block ends an item and the epilogue is waiting for it (56 vs 62 us).  Gating the early S on
            // "inputs already there" was slower in both cases.
            const bool s_first = cs.it < total_items && (cs.j != 0 || cp.nkb > 1);
            if (s_first) issue_s();
            const int st = gp & 1;
            ptx::mbar_wait(p_full, gp & 1);  // P of this block is in smem and O has been rescaled
            ptx::tc_fence_after();
            if (lane == 0) {
                const uint32_t p_base = ptx::smem_u32(sP);
                const uint32_t v_base = ptx::smem_u32(sKV + (size_t)st * 2 * KV_TILE_BYTES) + KV_TILE_BYTES;
#pragma unroll
                for (int k = 0; k < BKV / 16; ++k) {
                    const uint32_t a_addr = p_base + (k >> 2) * (BQ * 128) + (k & 3) * 32;
                    const uint32_t b_addr = v_base + k * 16 * 128;  // 16 keys = two 8-key swizzle atoms
                    ptx::umma_f16(tmem_base + O_COL, ptx::make_desc_k_sw128(a_addr),
                                  ptx::make_desc_mn_sw128(b_addr, 8192, 1024), idesc_o, (cp.j | k) != 0 ? 1u : 0u);
                }
                ptx::umma_commit(&kv_empty[st]);
                ptx::umma_commit(pv_done);
            }
            __syncwarp();
            ++gp;
            advance(cp, false);
            if (!s_first && cs.it < total_items) issue_s();
        }
    } else if (warp == 6 && BIAS) {
        // ================================================================== relative-bias row of each item's head
        // loaded into registers before waiting for the softmax warps to release the previous row, so the L2 latency
        // is hidden behind the previous item
        uint32_t n = 0;
        for (int it = blockIdx.x; it < total_items; it += gridDim.x, ++n) {
            const Item w = decode_item(it, q_blocks, H);
            const float* src = bias_log2 + (size_t)w.h * REL_T;
            float v[(REL_T + 31) / 32];
#pragma unroll
            for (int u = 0; u < (REL_T + 31) / 32; ++u) v[u] = lane + 32 * u < REL_T ? __ldg(src + lane + 32 * u) : 0.f;
            if (n > 0) ptx::mbar_wait(tail_empty, (n - 1) & 1);
#pragma unroll
            for (int u = 0; u < (REL_T + 31) / 32; ++u)
                if (lane + 32 * u < REL_T) sBias[lane + 32 * u] = v[u];
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(tail_full);
        }
    } else if (warp == 6) {
        // ================================================================== remainder key + remainder query row
        // (S = k * 128 + 1, e.g. the 257 tokens of ViT-L-14).  In every item this warp
        //   * scores the remainder KEY against the item's 128 query rows straight from the Q tile in shared memory and
        //     stages the scores + the key's V row for the softmax warps' epilogue (which then touches no global memory
        //     besides its output), and
        //   * is the second consumer of the K / V ring (kv_empty counts two arrivals);
        // in the items of the LAST query block it also computes the remainder ROW against the K / V tiles while they
        // sit in shared memory, with warp-level mma.sync (m16n8k16, row 0 of a 16-row tile) — a scalar version of this
        // took ~11 us per item and throttled the whole ring.
        uint32_t g = 0, n = 0, nt_staged = 0;   // key blocks, items, remainder-key stagings so far
        const size_t ld = (size_t)3 * W;
        const int gq = lane >> 2, tq = lane & 3;   // mma fragment coordinates: row group, column pair
        for (int it = blockIdx.x; it < total_items; it += gridDim.x, ++n) {
            const Item w = decode_item(it, q_blocks, H);
            int len, kend, nkb;
            item_extent<MASK, PACKED>(w, S, s_main, kv_len, len, kend, nkb, pack, B);
            const int row_base = w.b * stride;
            const bool do_row = inline_tail_rows > 0 && w.qb == q_blocks - 1;
            const int trow = s_main;   // the remainder row / key index
            ptx::mbar_wait(q_full, n & 1);
            if (s_main < len) {
                const __nv_bfloat16* krow = qkv + ((size_t)row_base + s_main) * ld + W + w.h * HD;
                uint4 k4[HD / 8];
#pragma unroll
                for (int u = 0; u < HD / 8; ++u) k4[u] = __ldg(reinterpret_cast<const uint4*>(krow) + u);
                const __nv_bfloat162 v2 = reinterpret_cast<const __nv_bfloat162*>(krow + W)[lane];
                {
                    const int nxt = it + gridDim.x;
                    if (lane == 0 && nxt < total_items) {   // the next item's remainder rows: into L2 ahead of time
                        const Item wn = decode_item(nxt, q_blocks, H);
                        const __nv_bfloat16* nrow = qkv + ((size_t)wn.b * stride + s_main) * ld + W + wn.h * HD;
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(nrow));
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(nrow + W));
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(nrow - W));
                    }
                }
                if (nt_staged > 0) ptx::mbar_wait(tail_empty, (nt_staged - 1) & 1);   // previous staging consumed
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int r = lane + 32 * i;
                    float acc = 0.f;
#pragma unroll
                    for (int u = 0; u < HD / 8; ++u) {
                        const uint4 q4 = *reinterpret_cast<const uint4*>(sQ + (size_t)r * 128 + ((u ^ (r & 7)) << 4));
                        const uint32_t qq[4] = {q4.x, q4.y, q4.z, q4.w};
                        const uint32_t kk[4] = {k4[u].x, k4[u].y, k4[u].z, k4[u].w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float2 qa = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&qq[e]));
                            const float2 ka = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&kk[e]));
                            acc = fmaf(qa.x, ka.x, acc);
                            acc = fmaf(qa.y, ka.y, acc);
                        }
                    }
                    sTailS[r] = acc * scale_log2e;
                }
                reinterpret_cast<__nv_bfloat162*>(sTailV)[lane] = v2;
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(tail_full);
                ++nt_staged;
            }
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(q_empty);   // this warp no longer needs the Q tile

            // ---- remainder row: A fragments of a 16-row tile whose row 0 is the query, rows 1..15 zero
            uint32_t qf[4][4];
            float o[8][4];
            float row_max = -INFINITY, row_sum = 0.f;   // row 0 lives in the lanes with gq == 0
            int tlimit = len;                           // keys >= tlimit are masked for the remainder row
            if (MASK == MASK_CAUSAL) tlimit = min(tlimit, trow + 1);
            if (do_row) {
                const __nv_bfloat16* qrow_p = qkv + ((size_t)row_base + trow) * ld + w.h * HD;
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
            }
            for (int j = 0; j < nkb; ++j, ++g) {
                const int st = g & 1;
                ptx::mbar_wait(&kv_full[st], (g >> 1) & 1);
                if (do_row) {
                    const __nv_bfloat16* kt = reinterpret_cast<const __nv_bfloat16*>(sKV + (size_t)st * 2 * KV_TILE_BYTES);
                    const __nv_bfloat16* vt = kt + BKV * HD;
                    const int mat = lane >> 3, rr8 = lane & 7;
                    auto tile_at = [](const __nv_bfloat16* tile, int row, int chunk) {
                        return tile + row * HD + ((chunk ^ (row & 7)) << 3);   // 128B-swizzled 16-byte chunks
                    };
                    // S = q K^T for the 128 keys of the block: 16 n-tiles of 8 keys
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
                    // mask + scale (log2 domain) + online softmax of row 0 (elements 0, 1 of every fragment)
                    float mx = row_max;
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int key = j * BKV + i * 8 + 2 * tq + e;
                            const float v = (key < tlimit && key < s_main) ? sc[i][e] * scale_log2e : -INFINITY;
                            sc[i][e] = v;
                            mx = fmaxf(mx, v);
                        }
                    }
                    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
                    const float msafe = mx == -INFINITY ? 0.f : mx;
                    const float corr = ex2(row_max - msafe);   // 0 on the first block
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
                            const float pv = ex2(sc[i][e] - msafe);   // exp2(-inf) = 0 for masked keys
                            ps += pv;
                            sc[i][e] = pv;
                        }
                    }
                    row_sum += ps;
                    // O += P V: 8 k-steps of 16 keys, 8 n-tiles of 8 dims; rows 8..15 of P are zero
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
                if (lane == 0) ptx::mbar_arrive(&kv_empty[st]);
            }
            if (do_row) {
                // the remainder key against the remainder row (global memory; lanes over the 64 dims, warp-reduced)
                if (s_main < tlimit) {
                    const __nv_bfloat16* qrow_p = qkv + ((size_t)row_base + trow) * ld + w.h * HD;
                    const __nv_bfloat16* krow = qkv + ((size_t)row_base + s_main) * ld + W + w.h * HD;
                    const float2 qpair = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(qrow_p)[lane]);
                    const float2 kf2 = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(krow)[lane]);
                    float sd = qpair.x * kf2.x + qpair.y * kf2.y;
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) sd += __shfl_xor_sync(0xffffffffu, sd, off);
                    const float scv = sd * scale_log2e;
                    const float m_new = fmaxf(row_max, scv);
                    const float alpha = ex2(row_max - m_new);
                    const float pe = ex2(scv - m_new);
                    const float pbv = __bfloat162float(__float2bfloat16_rn(pe));   // P is bf16 in the MMA path too
                    row_sum = row_sum * alpha + (tq == 0 ? pe : 0.f);               // row_sum is a per-quad partial
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
                    __nv_bfloat16* orow = out + ((size_t)row_base + trow) * W + w.h * HD;
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        *reinterpret_cast<uint32_t*>(orow + i * 8 + 2 * tq) = pack2(o[i][0] * inv_t, o[i][1] * inv_t);
                }
            }
        }
    } else {
        // ================================================================== softmax: thread == query row
        const int sp = warp & 3;
        const int r = sp * 32 + lane;  // row within the tile == TMEM lane
        const uint32_t lane_addr = tmem_base + (uint32_t(sp * 32) << 16);
        uint32_t g = 0, nt = 0;   // key blocks / remainder-key stagings consumed so far
        for (int it = blockIdx.x; it < total_items; it += gridDim.x) {
            const Item w = decode_item(it, q_blocks, H);
            int len, kend, nkb;
            item_extent<MASK, PACKED>(w, S, s_main, kv_len, len, kend, nkb, pack, B);
            const int row_base = w.b * stride;  // first row of this sequence / group in the packed [B*S, 3W] matrix
            const int qrow = w.q0 + r;     // position in the sequence (PACKED: row of the tile)
            const int h = w.h;
            // PACKED: this row's sequence inside the group and the keys it may see (block-diagonal mask)
            int p_lo = 0, p_hi = 0;
            bool row_valid = qrow < S;
            if (PACKED) {
                const int sidx = r / S;
                row_valid = sidx < pack && w.b * pack + sidx < B;
                if (row_valid) {
                    p_lo = sidx * S;
                    int n = S;
                    if (MASK == MASK_KEYLEN) n = min(S, max(kv_len[w.b * pack + sidx], 0));
                    p_hi = p_lo + n;
                    if (MASK == MASK_CAUSAL) p_hi = min(p_hi, r + 1);
                }
            }
            float m_run = -INFINITY, l_run = 0.f;
            // The remainder key (257 = 2 * 128 + 1) is folded in on the CUDA cores in the epilogue from the scores and
            // the V row that warp 6 stages in shared memory.
            const bool has_tail_key = !BIAS && s_main < len;   // uniform over the CTA
            const float* sB = nullptr;   // BIAS: the staged row at distance 0
            if constexpr (BIAS) {
                ptx::mbar_wait(tail_full, nt & 1);
                sB = sBias + REL_D;
            }
            const int tail_end = qrow < S ? (MASK == MASK_CAUSAL ? min(len, qrow + 1) : len) : 0;
            for (int j = 0; j < nkb; ++j, ++g) {
                const uint32_t par = g & 1;
                ptx::mbar_wait(s_full, par);
                ptx::tc_fence_after();
                int khi = kend - j * BKV;  // keys with block-local index outside [klo, khi) are masked
                if (MASK == MASK_CAUSAL) khi = min(khi, qrow - j * BKV + 1);
                int klo = 0;
                if (PACKED) {
                    klo = p_lo;
                    khi = p_hi;
                }
                const bool full = klo <= 0 && khi >= BKV;
                const int dk = j * BKV - qrow;   // BIAS: key - query of block-local key 0 (PACKED: tile rows = positions)
                // The exponent reference of a row is LAZY: it only moves when the block's true maximum exceeds it by
                // more than 2^8 (exp2(s - ref) <= 256 keeps P inside bf16's useful range and every sum far inside
                // fp32), so after a row's first block the O accumulator is almost never rescaled.  All decisions are
                // warp-uniform (__any_sync): tcgen05.ld / st are warp-collective.
                float lsum = 0.f, mx = -INFINITY, alpha = 1.f, m_new = m_run;
                uint32_t va[32];
                // ---- one pass: reference = running reference (first block: max of the row's first 32 scores); the
                //      exact maximum is tracked on the side and only checked afterwards
                ptx::tmem_ld_32x32b_x32(lane_addr + S_COL, va);
                tmem_ld_wait_regs(va);
                float m_ref = m_run;
                if (j == 0) {
                    float c0 = -INFINITY;
                    if constexpr (BIAS) {
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            if (full || (i >= klo && i < khi))
                                c0 = fmaxf(c0, fmaf(__uint_as_float(va[i]), scale_log2e, rel_bias(sB, dk + i)));
                        m_ref = c0;
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            if (full || (i >= klo && i < khi)) c0 = fmaxf(c0, __uint_as_float(va[i]));
                        m_ref = c0 * scale_log2e;
                    }
                }
                const float m_safe = m_ref == -INFINITY ? 0.f : m_ref;
                if (j > 0) ptx::mbar_wait(pv_done, par ^ 1);   // P buffer and O accumulator are free again
#pragma unroll 1
                for (int c = 0; c < BKV / 32; ++c) {
                    if (c > 0) {
                        ptx::tmem_ld_32x32b_x32(lane_addr + S_COL + c * 32, va);
                        tmem_ld_wait_regs(va);
                    }
                    if (full) softmax_chunk<true, BIAS>(va, c, klo, khi, scale_log2e, m_safe, lsum, mx, sP, r, sB, dk);
                    else softmax_chunk<false, BIAS>(va, c, klo, khi, scale_log2e, m_safe, lsum, mx, sP, r, sB, dk);
                }
                m_new = m_ref;
                const float m_true = fmaxf(m_ref, BIAS ? mx : mx * scale_log2e);
                const bool exceeded = m_true > m_safe + 8.0f;
                if (__any_sync(0xffffffffu, exceeded)) {
                    // exact update for this block: reference = true running maximum, P recomputed
                    m_new = m_true;
                    const float ms2 = m_new == -INFINITY ? 0.f : m_new;
                    alpha = ex2(m_run - ms2);   // 0 on the first block; 1 for rows whose reference did not move
                    lsum = 0.f;
                    float dummy = -INFINITY;
#pragma unroll 1
                    for (int c = 0; c < BKV / 32; ++c) {
                        ptx::tmem_ld_32x32b_x32(lane_addr + S_COL + c * 32, va);
                        tmem_ld_wait_regs(va);
                        if (full) softmax_chunk<true, BIAS>(va, c, klo, khi, scale_log2e, ms2, lsum, dummy, sP, r, sB, dk);
                        else softmax_chunk<false, BIAS>(va, c, klo, khi, scale_log2e, ms2, lsum, dummy, sP, r, sB, dk);
                    }
                }
                if (j == 0) alpha = 0.f;   // nothing accumulated yet (l_run == 0, O is overwritten by the first PV)
                l_run = l_run * alpha + lsum;
                m_run = m_new;
                // S has been consumed: the MMA warp may overwrite it with the next block's scores
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(s_free);
                if (j > 0 && __any_sync(0xffffffffu, alpha != 1.f)) {
                    // rescale the running output by alpha (thread-local: lane == row)
#pragma unroll 1
                    for (int c = 0; c < HD / 32; ++c) {
                        ptx::tmem_ld_32x32b_x32(lane_addr + O_COL + c * 32, va);
                        tmem_ld_wait_regs(va);
#pragma unroll
                        for (int i = 0; i < 32; ++i) va[i] = __float_as_uint(__uint_as_float(va[i]) * alpha);
                        ptx::tmem_st_32x32b_x32(lane_addr + O_COL + c * 32, va);
                    }
                    ptx::tmem_st_wait();
                }
                ptx::fence_proxy_async_smem();  // P (generic-proxy stores) -> visible to the tensor core's async proxy
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(p_full);
            }
            if constexpr (BIAS) {   // the scores of this item are done: warp 6 may stage the next item's row
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(tail_empty);
                ++nt;
            }
            // -------------------------------------------------------------- epilogue: (+ tail keys) O / l -> bf16
            // remainder key: online-softmax update of (m, l); the output is finished 32 dims at a time below
            float t_alpha = 1.f, t_p = 0.f;
            if (has_tail_key) {
                ptx::mbar_wait(tail_full, nt & 1);
                if (s_main < tail_end) {
                    const float sc = sTailS[r];
                    const float m_new = fmaxf(m_run, sc);
                    t_alpha = ex2(m_run - m_new);
                    const float pe = ex2(sc - m_new);
                    // the tensor-core path rounds P to bf16 before the PV product: do the same here
                    t_p = __bfloat162float(__float2bfloat16_rn(pe));
                    l_run = l_run * t_alpha + pe;
                    m_run = m_new;
                }
            }
            const float inv = l_run > 0.f ? 1.f / l_run : 0.f;
            if (nkb > 0) {
                ptx::mbar_wait(pv_done, (g - 1) & 1);
                ptx::tc_fence_after();
            }
#pragma unroll 1
            for (int hf = 0; hf < 2; ++hf) {
                float o[HD / 2];
                if (nkb > 0) {
                    uint32_t v0[32];
                    ptx::tmem_ld_32x32b_x32(lane_addr + O_COL + hf * 32, v0);
                    ptx::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) o[i] = __uint_as_float(v0[i]);
                } else {
#pragma unroll
                    for (int i = 0; i < HD / 2; ++i) o[i] = 0.f;
                }
                if (row_valid) {
                    if (has_tail_key) {   // o = o * alpha + p * v (alpha = 1, p = 0 for rows the key is masked for)
                        const uint4* vp = reinterpret_cast<const uint4*>(sTailV) + hf * 4;   // broadcast reads
#pragma unroll
                        for (int u = 0; u < HD / 16; ++u) {
                            const uint4 v4 = vp[u];
                            const uint32_t vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const float2 va = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&vv[e]));
                                o[8 * u + 2 * e] = fmaf(o[8 * u + 2 * e], t_alpha, t_p * va.x);
                                o[8 * u + 2 * e + 1] = fmaf(o[8 * u + 2 * e + 1], t_alpha, t_p * va.y);
                            }
                        }
                    }
                    uint4* d4 = reinterpret_cast<uint4*>(out + ((size_t)row_base + qrow) * W + h * HD) + hf * 4;
#pragma unroll
                    for (int u = 0; u < HD / 16; ++u) {
                        uint32_t pk[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            __nv_bfloat162 t2 = __floats2bfloat162_rn(o[8 * u + 2 * e] * inv, o[8 * u + 2 * e + 1] * inv);
                            pk[e] = *reinterpret_cast<uint32_t*>(&t2);
                        }
                        d4[u] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    }
                }
            }
            if (has_tail_key) {
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(tail_empty);
                ++nt;
            }
            // O has been read: order the tcgen05.ld before the p_full arrival that lets the next item's first PV
            // (accumulate = 0) overwrite it
            ptx::tc_fence_before();
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

}  // namespace tc

using KernelFn = void (*)(const CUtensorMap, const __nv_bfloat16*, __nv_bfloat16*, int, int, int, const int32_t*, float,
                          int, int, int, int, int, int, const float*);

// [bias][packed][mask]; no model combines the relative-position bias with causal masking (launch_tc rejects it)
static const KernelFn kernels[2][2][3] = {
    {{tc::attention_tc_kernel<MASK_NONE, false, false>, tc::attention_tc_kernel<MASK_CAUSAL, false, false>,
      tc::attention_tc_kernel<MASK_KEYLEN, false, false>},
     {tc::attention_tc_kernel<MASK_NONE, true, false>, tc::attention_tc_kernel<MASK_CAUSAL, true, false>,
      tc::attention_tc_kernel<MASK_KEYLEN, true, false>}},
    {{tc::attention_tc_kernel<MASK_NONE, false, true>, nullptr, tc::attention_tc_kernel<MASK_KEYLEN, false, true>},
     {tc::attention_tc_kernel<MASK_NONE, true, true>, nullptr, tc::attention_tc_kernel<MASK_KEYLEN, true, true>}}};

int launch_tc(const __nv_bfloat16* qkv, __nv_bfloat16* out, int B, int S, int W, int H, int mask, const int32_t* kv_len,
              const float* bias_log2, cudaStream_t stream) {
    if (B <= 0 || S <= 0) return 0;
    if (W != H * tc::HD) fail(B200_ERR_UNSUPPORTED, "attention: head_dim must be 64 (width %d, heads %d)", W, H);
    if (mask < MASK_NONE || mask > MASK_KEYLEN) fail(B200_ERR_INTERNAL, "attention: unknown mask mode %d", mask);
    if (mask == MASK_KEYLEN && !kv_len) fail(B200_ERR_INTERNAL, "attention: kv_len required for key-length masking");
    const bool bias = bias_log2 != nullptr;
    if (bias && mask == MASK_CAUSAL)
        fail(B200_ERR_INTERNAL, "attention: causal masking takes no relative-position bias");
    const uint32_t smem = bias ? tc::SMEM_BYTES_BIAS : tc::SMEM_BYTES;
    static std::once_flag once;
    std::call_once(once, [] {
        for (int bs = 0; bs < 2; ++bs)
            for (int pk = 0; pk < 2; ++pk)
                for (int mk = 0; mk < 3; ++mk)
                    if (kernels[bs][pk][mk])
                        MB_CUDA(cudaFuncSetAttribute(kernels[bs][pk][mk], cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                     (int)(bs ? tc::SMEM_BYTES_BIAS : tc::SMEM_BYTES)));
    });
    // one tensor map over the packed [B*S, 3W] matrix serves Q, K and V tiles (64 columns x 128 rows, 128B swizzle);
    // rows past the end of the matrix are zero-filled, rows of the next sequence are masked by key index
    CUtensorMap tmap = make_tmap_2d(qkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)3 * W, (uint64_t)B * S,
                                    (uint64_t)3 * W * 2, tc::HD, tc::BQ, CU_TENSOR_MAP_SWIZZLE_128B);
    const float scale_log2e = 0.125f * 1.4426950408889634f;
    int device = 0;
    MB_CUDA(cudaGetDevice(&device));
    if (S < tc::BQ) {
        // Short sequences (ViT-B-32: 50 tokens, CLIP text: 77, short BERT batches): pack = 128 / S whole sequences share
        // one 128 x 128 tile under a block-diagonal mask — S = 50 fills 100 of the 128 rows instead of 50.
        const int pack = tc::BQ / S;
        const int groups = (B + pack - 1) / pack;
        const int total_items = groups * H;
        const int grid = std::min(2 * sm_count(device), total_items);
        kernels[bias][1][mask]<<<grid, tc::THREADS, smem, stream>>>(
            tmap, qkv, out, S, W, H, kv_len, scale_log2e, /*s_main=*/1 << 30, 0, /*q_blocks=*/1, total_items, pack, B,
            bias_log2);
        MB_CUDA(cudaGetLastError());
        return 1;
    }
    // A remainder of ONE token (S = 257, 129, ...: a class token on top of a power-of-two grid) is not worth a 128-wide
    // tile in either dimension: warp 6 of the kernel handles that key and that query row.  The bias variants use warp 6
    // and the remainder's shared memory for the bias row instead and run such a sequence as one more masked block.
    const int rem = S % tc::BQ;
    const bool tail = !bias && S > tc::BQ && rem == 1;
    const int s_main = tail ? S - rem : S;                       // keys handled by the tensor cores
    const int q_blocks = tail ? S / tc::BQ : (S + tc::BQ - 1) / tc::BQ;
    const int inline_rows = tail ? rem : 0;
    // persistent grid: two CTAs per SM; an odd CTA count when q_blocks is even makes every CTA alternate between the
    // query blocks of a sequence, so the remainder-row work of the last block is spread over all CTAs
    const int total_items = B * H * q_blocks;
    int grid = 2 * sm_count(device);
    if ((q_blocks & 1) == 0 && (grid & 1) == 0) grid -= 1;
    grid = std::min(grid, total_items);
    kernels[bias][0][mask]<<<grid, tc::THREADS, smem, stream>>>(
        tmap, qkv, out, S, W, H, kv_len, scale_log2e, s_main, inline_rows, q_blocks, total_items, 1, B, bias_log2);
    MB_CUDA(cudaGetLastError());
    return 1;
}

}  // namespace attention
}  // namespace mb
