// K2 -- batched query x embedding similarity on the 5th-gen tensor cores (tcgen05, sm_100a).
//
// Replaces the per-query fp32 sgemv of get_fact_scores / dense_passage_retrieval (reference
// HippoRAG.py:1459, :1496: np.dot(E, q)) with one batched contraction S = Q E^T:
//   D[128 queries, 256 embeddings] (fp32, TMEM) += A[128, 64] (bf16, smem) * B[256, 64]^T (bf16, smem)
// Both operands are K-major (a row = one embedding), staged by TMA (128-byte swizzle) into a
// 4-stage shared-memory ring; one elected thread issues tcgen05.mma; accumulators live in TMEM,
// double-buffered (2 x 256 columns) so the epilogue of tile t overlaps the MMAs of tile t+1.
//
// Precision (SURVEY.md 7, hard part 3): a single bf16 pass flips top-k membership, so the parity
// mode is the fp32-faithful split  x = hi + lo (both bf16, 16 mantissa bits together):
//     q.e ~= q_lo.e_lo + q_hi.e_lo + q_lo.e_hi + q_hi.e_hi      (fp32 accumulate in TMEM)
// All four products are issued per k-block from ONE stage holding {q_hi, q_lo, e_hi, e_lo}:
// 4 products per byte-set of operand traffic, where three separate K-passes would move 1.5x the
// bytes for 3.  Split stages are 32 K-columns wide (64-byte swizzle, 48 KB, 4 stages) so three
// TMA batches are in flight while one is consumed (2 x 96-KB stages left the MMA issuer waiting
// on load latency: ncu 39 % tensor pipe, profiles/r1_k2_sim_tc_ncu.md).  The lo.lo term is kept because it is systematic (always positive)
// exactly for the highly correlated query/fact pairs that end up in the top-k.
// HRAG_SIM_BF16 = hi.hi only (48 KB stages, 4 of them).
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..5 = epilogue (TMEM -> registers -> global, one query row per thread).
#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>

#include "common.cuh"
#include "kernels.h"

namespace hrag {

namespace {

constexpr int BM = 128;          // queries per tile  (UMMA M)
constexpr int BN = 256;          // embeddings per tile (UMMA N)
constexpr int BK = 64;           // bf16 elements per k-block = one 128-byte swizzle row
constexpr int UK = 16;           // UMMA K for 16-bit inputs
constexpr int RING_BYTES = 4 * (BM + BN) * BK * 2;   // 192 KB = 4 stages of 48 KB in both modes
constexpr int TMEM_COLS = 512;                 // 2 accumulators x 256 fp32 columns
constexpr int TC_THREADS = 192;
constexpr size_t SMEM_BYTES = (size_t)RING_BYTES + 1024 /*align*/ + 256 /*barriers*/;

// ---- PTX wrappers ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* map, int c0, int c1) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(map), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols));
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread = TMEM lane = query row)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA shared-memory descriptor of a K-major operand tile whose rows are ROW_BYTES wide
// (128 -> SWIZZLE_128B, 64 -> SWIZZLE_64B): 8-row swizzle atoms 8*ROW_BYTES apart (SBO); LBO unused
// for these layouts; descriptor version 1 (sm_100).
template <int ROW_BYTES>
__device__ __forceinline__ uint64_t umma_desc_kmajor(uint32_t smem_addr) {
    static_assert(ROW_BYTES == 128 || ROW_BYTES == 64, "row = one swizzle span");
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);        // start address, 16-byte units
    d |= (uint64_t)((8u * ROW_BYTES) >> 4) << 32;        // stride byte offset
    d |= (uint64_t)1 << 46;                              // version
    d |= (uint64_t)(ROW_BYTES == 128 ? 2 : 4) << 61;     // layout: SWIZZLE_128B = 2, SWIZZLE_64B = 4
    return d;
}
// Instruction descriptor, kind::f16: D fp32, A/B bf16, both K-major, M = 128, N = 256.
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) |
                            ((uint32_t)(BM >> 4) << 24);

struct TcParams {
    int Bq;            // valid query rows
    int64_t M;         // valid embedding rows
    int dim;
    float* S;
    int64_t ldS;
    int num_m_tiles, num_n_tiles;
    // fused epilogue (FUSE): per (query, n-tile) min/max and the 8 best rank keys instead of scores
    float2* part_mm;          // [Bq, num_n_tiles]
    uint64_t* part_keys;      // [Bq, num_n_tiles, 8]
    // threshold epilogue (FUSE == 2, index-time synonymy KNN): every score >= thr is appended to its query's
    // candidate list as a rank key; cand_count keeps counting past cand_cap so overflow is detectable
    float thr;
    uint64_t* cand_keys;      // [Bq, cand_cap]
    int* cand_count;          // [Bq]
    int cand_cap;
};

constexpr int kFuseK = 8;

template <bool SPLIT, int FUSE>          // FUSE: 0 = store scores, 1 = min/max + 8 best per tile, 2 = threshold append
__global__ void __launch_bounds__(TC_THREADS, 1)
k_sim_tc(const __grid_constant__ CUtensorMap map_q_hi, const __grid_constant__ CUtensorMap map_q_lo,
         const __grid_constant__ CUtensorMap map_e_hi, const __grid_constant__ CUtensorMap map_e_lo, TcParams p) {
    constexpr int STAGES = 4;
    constexpr int BKs = SPLIT ? BK / 2 : BK;                 // K-columns per stage
    constexpr int ROW_BYTES = BKs * 2;                       // = the TMA / UMMA swizzle span
    constexpr int A_BYTES = BM * ROW_BYTES, B_BYTES = BN * ROW_BYTES;
    constexpr int STAGE_BYTES = (SPLIT ? 2 : 1) * (A_BYTES + B_BYTES);   // 48 KB either way
    // stage layout: [A_hi | B_hi] or [A_hi | A_lo | B_hi | B_lo]
    constexpr int OFF_A_LO = A_BYTES, OFF_B_HI = SPLIT ? 2 * A_BYTES : A_BYTES, OFF_B_LO = 2 * A_BYTES + B_BYTES;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;                 // SWIZZLE_128B tiles need 1024-B alignment
    const uint32_t bars = base + RING_BYTES;                      // barrier block
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 64u + 8u * s; };
    auto tfull_bar = [&](int a) { return bars + 128u + 8u * a; };
    auto tempty_bar = [&](int a) { return bars + 160u + 8u * a; };
    const uint32_t tmem_slot = bars + 192u;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nkb = (p.dim + BKs - 1) / BKs;
    const int total_tiles = p.num_m_tiles * p.num_n_tiles;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_q_hi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_e_hi) : "memory");
        if (SPLIT) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_q_lo) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_e_lo) : "memory");
        }
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
            for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        tmem_alloc(tmem_slot, TMEM_COLS);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const int mt = t % p.num_m_tiles, nt = t / p.num_m_tiles;
                // L2 prefetch of this CTA's share of the NEXT embedding tile: the num_m_tiles CTAs that
                // will work on it each pull every num_m_tiles-th k-block, a whole tile ahead, so the
                // later TMA loads are L2 hits (ncu before: 3x algorithmic DRAM reads, 39 % tensor pipe)
                const int tn = t + gridDim.x;
                if (tn < total_tiles) {
                    const int mtn = tn % p.num_m_tiles, ntn = tn / p.num_m_tiles;
                    for (int kb = mtn; kb < nkb; kb += p.num_m_tiles) {
                        tma_prefetch_l2_2d(&map_e_hi, kb * BKs, ntn * BN);
                        if (SPLIT) tma_prefetch_l2_2d(&map_e_lo, kb * BKs, ntn * BN);
                    }
                }
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait(empty_bar(stage), phase ^ 1u);
                    mbar_expect_tx(full_bar(stage), STAGE_BYTES);
                    const uint32_t sa = base + stage * STAGE_BYTES;
                    tma_load_2d(sa, &map_q_hi, full_bar(stage), kb * BKs, mt * BM);
                    tma_load_2d(sa + OFF_B_HI, &map_e_hi, full_bar(stage), kb * BKs, nt * BN);
                    if (SPLIT) {
                        tma_load_2d(sa + OFF_A_LO, &map_q_lo, full_bar(stage), kb * BKs, mt * BM);
                        tma_load_2d(sa + OFF_B_LO, &map_e_lo, full_bar(stage), kb * BKs, nt * BN);
                    }
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one thread) =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                mbar_wait(tempty_bar(acc), acc_phase ^ 1u);     // epilogue drained this accumulator
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t sa = base + stage * STAGE_BYTES;
                    const uint64_t a_hi = umma_desc_kmajor<ROW_BYTES>(sa), b_hi = umma_desc_kmajor<ROW_BYTES>(sa + OFF_B_HI);
                    if (SPLIT) {
                        const uint64_t a_lo = umma_desc_kmajor<ROW_BYTES>(sa + OFF_A_LO);
                        const uint64_t b_lo = umma_desc_kmajor<ROW_BYTES>(sa + OFF_B_LO);
                        // smallest terms first: lo.lo, hi.lo, lo.hi, then hi.hi
#pragma unroll
                        for (int k = 0; k < BKs / UK; ++k)
                            umma_bf16(tmem_d, a_lo + (uint64_t)(2 * k), b_lo + (uint64_t)(2 * k), kIdesc,
                                      (kb > 0 || k > 0) ? 1u : 0u);
#pragma unroll
                        for (int k = 0; k < BKs / UK; ++k)
                            umma_bf16(tmem_d, a_hi + (uint64_t)(2 * k), b_lo + (uint64_t)(2 * k), kIdesc, 1u);
#pragma unroll
                        for (int k = 0; k < BKs / UK; ++k)
                            umma_bf16(tmem_d, a_lo + (uint64_t)(2 * k), b_hi + (uint64_t)(2 * k), kIdesc, 1u);
#pragma unroll
                        for (int k = 0; k < BKs / UK; ++k)
                            umma_bf16(tmem_d, a_hi + (uint64_t)(2 * k), b_hi + (uint64_t)(2 * k), kIdesc, 1u);
                    } else {
#pragma unroll
                        for (int k = 0; k < BKs / UK; ++k)   // +32 bytes (2 x 16-byte units) along K per step
                            umma_bf16(tmem_d, a_hi + (uint64_t)(2 * k), b_hi + (uint64_t)(2 * k), kIdesc,
                                      (kb > 0 || k > 0) ? 1u : 0u);
                    }
                    umma_commit(empty_bar(stage));               // smem slot free once these MMAs retire
                    if (kb == nkb - 1) umma_commit(tfull_bar(acc));
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
                if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
            }
        }
    } else {
        // ===== epilogue: warps 2..5, TMEM lane quarter = warp % 4 =====
        const int quarter = warp & 3;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const int mt = t % p.num_m_tiles, nt = t / p.num_m_tiles;
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
            const int q = mt * BM + quarter * 32 + lane;
            const int64_t n0 = (int64_t)nt * BN;
            if (FUSE == 2) {
                // this thread owns query q: every score of the tile that clears the threshold joins q's candidate list
#pragma unroll 1
                for (int c = 0; c < BN / 32; ++c) {
                    uint32_t r[32];
                    tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + c * 32), r);
                    if (q < p.Bq) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int64_t col = n0 + c * 32 + j;
                            const float f = __uint_as_float(r[j]);
                            if (col < p.M && f >= p.thr) {
                                const int pos = atomicAdd(p.cand_count + q, 1);
                                if (pos < p.cand_cap) p.cand_keys[(size_t)q * p.cand_cap + pos] = rank_key(f, (uint32_t)col);
                            }
                        }
                    }
                }
            } else if (FUSE == 1) {
                // this thread owns query q: scan the tile's 256 scores once, keep min / max / 8 best
                float mn = INFINITY, mx = -INFINITY;
                uint64_t best[kFuseK];
#pragma unroll
                for (int j = 0; j < kFuseK; ++j) best[j] = 0ull;
#pragma unroll 1
                for (int c = 0; c < BN / 32; ++c) {
                    uint32_t r[32];
                    tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + c * 32), r);
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int64_t col = n0 + c * 32 + j;
                        if (col < p.M) {
                            const float f = __uint_as_float(r[j]);
                            mn = fminf(mn, f);
                            mx = fmaxf(mx, f);
                            uint64_t key = rank_key(f, (uint32_t)col);
                            if (key > best[kFuseK - 1]) {
#pragma unroll
                                for (int k = 0; k < kFuseK; ++k)
                                    if (key > best[k]) { const uint64_t tmp = best[k]; best[k] = key; key = tmp; }
                            }
                        }
                    }
                }
                if (q < p.Bq) {
                    const size_t o = (size_t)q * p.num_n_tiles + nt;
                    p.part_mm[o] = make_float2(mn, mx);
#pragma unroll
                    for (int k = 0; k < kFuseK; k += 2)
                        *reinterpret_cast<ulonglong2*>(p.part_keys + o * kFuseK + k) = make_ulonglong2(best[k], best[k + 1]);
                }
            } else {
            float* row = p.S + (size_t)q * p.ldS + n0;
#pragma unroll 1
            for (int c = 0; c < BN / 32; ++c) {
                uint32_t r[32];
                tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + c * 32), r);
                if (q < p.Bq) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        if (n0 + c * 32 + j < p.ldS)     // ldS is a multiple of 4: whole float4 in range
                            *reinterpret_cast<float4*>(row + c * 32 + j) =
                                make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                            __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
                    }
                }
            }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(acc));
            if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// x = hi + lo with hi = bf16(x), lo = bf16(x - hi)
__global__ void __launch_bounds__(256)
k_split_bf16(const float* __restrict__ x, int64_t n, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
    const int64_t i = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 4;
    if (i >= n) return;
    if (i + 3 < n) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(x + i));
        const float f[4] = {v.x, v.y, v.z, v.w};
        __nv_bfloat16 h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            h[j] = __float2bfloat16_rn(f[j]);
            l[j] = __float2bfloat16_rn(f[j] - __bfloat162float(h[j]));
        }
        *reinterpret_cast<uint2*>(hi + i) = *reinterpret_cast<uint2*>(h);
        *reinterpret_cast<uint2*>(lo + i) = *reinterpret_cast<uint2*>(l);
    } else {
        for (int64_t j = i; j < n; ++j) {
            const __nv_bfloat16 h = __float2bfloat16_rn(x[j]);
            hi[j] = h;
            lo[j] = __float2bfloat16_rn(x[j] - __bfloat162float(h));
        }
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;

int get_encoder() {
    if (g_encode) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    HRAG_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    HRAG_CHECK(fn != nullptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    return 0;
}

// [rows, dim] bf16 row-major -> 2-D tensor map with a {box_cols x box_rows} box whose row is one
// swizzle span (64 columns -> 128-byte swizzle, 32 -> 64-byte swizzle).
int make_map(CUtensorMap* map, const void* ptr, int64_t rows, int dim, int box_cols, int box_rows) {
    HRAG_TRY(get_encoder());
    cuuint64_t gdim[2] = {(cuuint64_t)dim, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)dim * 2};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estride[2] = {1, 1};
    CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box,
                          estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    HRAG_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
    return 0;
}

}  // namespace

int split_bf16(const float* x, int64_t n, void* hi, void* lo, cudaStream_t stream) {
    if (n == 0) return 0;
    k_split_bf16<<<(unsigned)ceil_div(ceil_div(n, 4), 256), 256, 0, stream>>>(
        x, n, reinterpret_cast<__nv_bfloat16*>(hi), reinterpret_cast<__nv_bfloat16*>(lo));
    count_launch(1);
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

int sim_tc_n_tiles(int64_t M) { return (int)ceil_div(M, BN); }

int sim_tc_threshold(const void* q_hi, const void* q_lo, int Bq, const void* e_hi, const void* e_lo, int64_t M, int dim,
                     int n_seg, float thr, uint64_t* cand_keys, int* cand_count, int cand_cap, int num_sms,
                     cudaStream_t stream) {
    HRAG_CHECK(dim % 8 == 0, "sim_tc: embedding dim must be a multiple of 8 (TMA row pitch)");
    HRAG_CHECK(n_seg == 1 || n_seg == 4, "sim_tc: n_seg must be 1 (bf16) or 4 (split)");
    HRAG_CHECK(cand_keys && cand_count && cand_cap > 0, "sim_tc_threshold: candidate buffers missing");
    if (Bq == 0 || M == 0) return 0;
    static bool attr_set = false;
    if (!attr_set) {
        HRAG_CUDA(cudaFuncSetAttribute(k_sim_tc<true, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        HRAG_CUDA(cudaFuncSetAttribute(k_sim_tc<false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        attr_set = true;
    }
    CUtensorMap mqh, mql, meh, mel;
    const int bkc = n_seg == 4 ? BK / 2 : BK;
    HRAG_TRY(make_map(&mqh, q_hi, Bq, dim, bkc, BM));
    HRAG_TRY(make_map(&mql, q_lo, Bq, dim, bkc, BM));
    HRAG_TRY(make_map(&meh, e_hi, M, dim, bkc, BN));
    HRAG_TRY(make_map(&mel, e_lo, M, dim, bkc, BN));
    TcParams p;
    p.Bq = Bq; p.M = M; p.dim = dim; p.S = nullptr; p.ldS = 0; p.part_mm = nullptr; p.part_keys = nullptr;
    p.thr = thr; p.cand_keys = cand_keys; p.cand_count = cand_count; p.cand_cap = cand_cap;
    p.num_m_tiles = (int)ceil_div(Bq, BM);
    p.num_n_tiles = (int)ceil_div(M, BN);
    const int grid = (int)std::min<int64_t>((int64_t)p.num_m_tiles * p.num_n_tiles, num_sms);
    if (n_seg == 4) k_sim_tc<true, 2><<<grid, TC_THREADS, SMEM_BYTES, stream>>>(mqh, mql, meh, mel, p);
    else k_sim_tc<false, 2><<<grid, TC_THREADS, SMEM_BYTES, stream>>>(mqh, mql, meh, mel, p);
    count_launch(1);
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

int sim_tc(const void* q_hi, const void* q_lo, int Bq, const void* e_hi, const void* e_lo, int64_t M, int dim,
           int n_seg, float* S, int64_t ldS, float2* part_mm, uint64_t* part_keys, int num_sms, cudaStream_t stream) {
    HRAG_CHECK(dim % 8 == 0, "sim_tc: embedding dim must be a multiple of 8 (TMA row pitch)");
    HRAG_CHECK(n_seg == 1 || n_seg == 4, "sim_tc: n_seg must be 1 (bf16) or 4 (split)");
    if (Bq == 0 || M == 0) return 0;
    static bool attr_set = false;
    if (!attr_set) {
        HRAG_CUDA(cudaFuncSetAttribute(k_sim_tc<true, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        HRAG_CUDA(cudaFuncSetAttribute(k_sim_tc<false, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        HRAG_CUDA(cudaFuncSetAttribute(k_sim_tc<true, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        HRAG_CUDA(cudaFuncSetAttribute(k_sim_tc<false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        attr_set = true;
    }
    CUtensorMap mqh, mql, meh, mel;
    const int bkc = n_seg == 4 ? BK / 2 : BK;
    HRAG_TRY(make_map(&mqh, q_hi, Bq, dim, bkc, BM));
    HRAG_TRY(make_map(&mql, q_lo, Bq, dim, bkc, BM));
    HRAG_TRY(make_map(&meh, e_hi, M, dim, bkc, BN));
    HRAG_TRY(make_map(&mel, e_lo, M, dim, bkc, BN));
    TcParams p;
    p.Bq = Bq; p.M = M; p.dim = dim; p.S = S; p.ldS = ldS; p.part_mm = part_mm; p.part_keys = part_keys;
    const bool fuse = part_mm != nullptr;
    p.thr = 0.f; p.cand_keys = nullptr; p.cand_count = nullptr; p.cand_cap = 0;
    HRAG_CHECK(fuse || (S != nullptr && ldS % 4 == 0), "sim_tc: score buffer missing");
    p.num_m_tiles = (int)ceil_div(Bq, BM);
    p.num_n_tiles = (int)ceil_div(M, BN);
    const int grid = (int)std::min<int64_t>((int64_t)p.num_m_tiles * p.num_n_tiles, num_sms);
    if (n_seg == 4 && fuse) k_sim_tc<true, 1><<<grid, TC_THREADS, SMEM_BYTES, stream>>>(mqh, mql, meh, mel, p);
    else if (n_seg == 4) k_sim_tc<true, 0><<<grid, TC_THREADS, SMEM_BYTES, stream>>>(mqh, mql, meh, mel, p);
    else if (fuse) k_sim_tc<false, 1><<<grid, TC_THREADS, SMEM_BYTES, stream>>>(mqh, mql, meh, mel, p);
    else k_sim_tc<false, 0><<<grid, TC_THREADS, SMEM_BYTES, stream>>>(mqh, mql, meh, mel, p);
    count_launch(1);
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace hrag
