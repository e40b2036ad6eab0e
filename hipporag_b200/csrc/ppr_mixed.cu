// K1m -- mixed-precision PPR: fp16 state, fp32 arithmetic, iterative refinement.
//
// K1 (ppr_spmm.cu) is bound by the rate at which the SMs can pull gathered rows of the state
// matrix out of L2 (DESIGN.md section 4), i.e. by bytes per gathered row.  Storing the iterate
// in fp16 halves those bytes: a [N, 32] fp16 state has the same 64-byte rows as the [N, 16]
// fp32 state, so one sweep costs the same and serves twice the queries.  fp32-level accuracy is
// recovered by classical iterative refinement on the linear system (I - aP) x = v:
//     1. x0  ~ solve(v)          m1 Chebyshev sweeps, state + rhs in fp16 (scaled per column)
//     2. r   = v - x0 + aP x0    ONE sweep, fp32 arithmetic on the exact fp32 v and the fp16 x0
//     3. d   ~ solve(r)          m2 Chebyshev sweeps in fp16 (r scaled by t)
//     4. x   = x0 + d            only where it is consumed (passage rows) + the column sums
// (when one round cannot reach the requested tolerance -- large damping -- the caller takes the fp32
// solver instead, api.cu plan_sweeps).  Every product is accumulated in fp32; only the STORED
// iterate is rounded, and step 2 measures exactly what that rounding (and the truncated step 1)
// left behind: its column sums give the residual check of the solve for free.
//
// Layout: half state [N, 32] row-major (64 B per row); a group of 4 lanes owns a row, each lane
// 8 columns (one 16-byte load per gathered row per lane).  Rows > long_thresh use the same
// segment scheme as K1.
//
// Right-hand side.  The reset vector of graph_search_with_fact_entities (HippoRAG.py:1544-1656)
// is non-zero only on the P passage vertices and on <= link_top_k phrase vertices per query, so
// it is kept COMPACT: `slot_map[node]` (-1 = the row has no rhs) points into `[n_slots, 32]`
// arrays (fp32 exact v, fp16 scaled rhs).  The 90 % of rows that are neither passages nor seeds
// read 4 bytes instead of 64, and building the rhs of a sub-batch touches P x 32 values instead
// of three passes over [N, 32] fp32.  slot_map == nullptr means "dense": slot = row (hrag_ppr's
// arbitrary reset vectors, and the residual rhs of the correction solve).
//
// Row walk: 4 gathers in flight per lane, the ragged end of a row is one PREDICATED batch (not a
// serial tail), and the 64 rows of a CTA are handed to the groups by length (row_order) so the 8
// rows that share a warp finish together.  Loads are plain read-only loads: cache-policy
// descriptors on gathers / streams and L1::no_allocate were measured slower once the tail is
// predicated -- profiles/r2_k1m_variants_{a,b,c}.txt.
//
// K5 (node-range sharding, k_sweep_h_push): each CTA stages its 64 output rows in shared memory
// and pushes the 4-KB block into every peer GPU's copy of y with one TMA bulk copy per peer over
// NVLink; the epoch handshake that replaces a collective is folded into the sweep itself: every
// CTA starts by polling the local flag words (ld.relaxed.sys), the last CTA of the persistent
// grid to finish publishes this rank's epoch to the peers (st.release.sys) -- no extra launches.
#include <cuda_fp16.h>

#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"

namespace hrag {

namespace {

constexpr int kThreads = 256;
constexpr int kLPR = 4;                 // lanes per row
constexpr int kGPB = kThreads / kLPR;   // rows per CTA
constexpr int kB = 32;                  // batch width of the mixed solver

__device__ __forceinline__ void h8_to_f(const uint4& u, float (&f)[8]) {
    const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float2 a = __half22float2(h[j]);
        f[2 * j] = a.x;
        f[2 * j + 1] = a.y;
    }
}
__device__ __forceinline__ float sat_h(float x) { return fminf(fmaxf(x, -65504.f), 65504.f); }
__device__ __forceinline__ uint4 f_to_h8(const float (&f)[8]) {
    uint4 u;
    __half2* h = reinterpret_cast<__half2*>(&u);
#pragma unroll
    for (int j = 0; j < 4; ++j) h[j] = __floats2half2_rn(sat_h(f[2 * j]), sat_h(f[2 * j + 1]));
    return u;
}
__device__ __forceinline__ void fma8(float (&acc)[8], float a, const uint4& u) {
    float f[8];
    h8_to_f(u, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = fmaf(a, f[j], acc[j]);
}

// ---- loads ----------------------------------------------------------------------------------------
// predicated: `ok == false` yields zeros without touching memory (the ragged end of a row is a predicated batch)
__device__ __forceinline__ uint4 ld_gather(const uint4* p, bool ok) { return ok ? __ldg(p) : make_uint4(0u, 0u, 0u, 0u); }
__device__ __forceinline__ int2 ld_cv(const int2* p, bool ok) { return ok ? __ldg(p) : make_int2(0, 0); }
// read-once operand of the epilogue (rhs, exact v): streamed, first out of the caches
__device__ __forceinline__ uint4 ld_stream16(const void* p) { return __ldcs(reinterpret_cast<const uint4*>(p)); }
// prev may alias y (in-place Chebyshev): a coherent load, no .nc.  A copy, not a reference into global memory:
// handing h8_to_f the reference directly schedules the sweep's epilogue differently
__device__ __forceinline__ uint4 ld_prev(const uint4* p) { return *p; }

template <int U>
__device__ __forceinline__ void group_row_dot_h(const int2* __restrict__ cv, int s, int e,
                                                const uint4* __restrict__ xh /* + lane */, float (&acc)[8]) {
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    // U independent 16-byte gathers in flight per lane; the ragged end of the row is a PREDICATED batch, not a
    // serial one-at-a-time loop (a row of 14 non-zeros costs 4 round trips to L2, not 3 + 2)
    for (int i = s; i < e; i += U) {
        int2 c[U];
        uint4 a[U];
#pragma unroll
        for (int j = 0; j < U; ++j) c[j] = ld_cv(cv + i + j, i + j < e);
#pragma unroll
        for (int j = 0; j < U; ++j) a[j] = ld_gather(xh + (size_t)c[j].x * kLPR, i + j < e);
#pragma unroll
        for (int j = 0; j < U; ++j) fma8(acc, __int_as_float(c[j].y), a[j]);
    }
}

// ---- K5 epoch handshake, folded into the sweep kernels ---------------------------------------
__device__ __forceinline__ void sync_wait(const SweepSync& sy) {
    if (sy.flags == nullptr) return;                 // single GPU (uniform branch)
    const int r = threadIdx.x;
    if (r < sy.world && r != sy.rank) {
        unsigned long long v = 0;
        long long spin = 0;
#pragma unroll 1
        for (; spin < (1ll << 24); ++spin) {         // bounded (~seconds): a lost peer must not hang the GPU
            // relaxed, not acquire: an acquire load at system scope is followed by CCTL.IVALL, i.e. every poll of every
            // CTA would flush the SM's L1 under the CTAs already gathering.  Nothing stale can be in L1: it is
            // invalidated at kernel launch and no row of x is loaded before this wait has passed.
            asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(sy.flags + r) : "memory");
            if (v >= sy.need) break;
            __nanosleep(32);
        }
        if (v < sy.need) *sy.error_flag = 1;
    }
    __syncthreads();
}
__device__ __forceinline__ void sync_signal(const SweepSync& sy) {
    if (sy.flags == nullptr || sy.done_ctr == nullptr) return;
    __syncthreads();                                 // every thread's (peer) stores are issued
    if (threadIdx.x == 0) {
        if (!(sy.debug & 1)) __threadfence_system();
        const unsigned int prev = atomicAdd(sy.done_ctr, 1u);
        if (prev + 1 == sy.total_ctas) {             // last CTA of the sweep: publish this rank's epoch
            *sy.done_ctr = 0;
            __threadfence_system();
#pragma unroll
            for (int i = 0; i < 7; ++i)                  // static indices: kernel parameters stay in the constant bank
                if (i < sy.n_remote)
                    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(sy.remote[i]), "l"(sy.epoch) : "memory");
        }
    }
}

// MODE 0: y = w * (alpha * acc + rhs) + (1 - w) * prev        (all fp16 in memory)
// MODE 1: y = t * (scale * v32 - x0 + alpha * acc)            (the refinement residual)
// rhs / v32 are addressed through slot_map (null = dense).  Returns (in out[]) the value as
// STORED (after fp16 rounding) so column sums match memory; MODE 1 + FINAL returns |value|.
template <bool CHEB, int MODE>
__device__ __forceinline__ void row_epilogue_h(float (&acc)[8], int row, int lane, const int* __restrict__ slot_map,
                                               const uint4* __restrict__ rhs_h, const float4* __restrict__ v32,
                                               const float* __restrict__ col_scale, const uint4* x0h,
                                               const uint4* prevh, uint4* yh, float alpha, float w, float t,
                                               const PeerOut& peers, float (&out)[8], uint4& packed_out) {
    const size_t o = (size_t)row * kLPR + lane;
    const int slot = slot_map ? __ldg(slot_map + row) : row;
    if (MODE == 0) {
        if (slot >= 0) {
            float r[8];
            h8_to_f(ld_stream16(rhs_h + (size_t)slot * kLPR + lane), r);
#pragma unroll
            for (int j = 0; j < 8; ++j) out[j] = fmaf(alpha, acc[j], r[j]);
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) out[j] = alpha * acc[j];
        }
        if (CHEB) {
            float p[8];
            h8_to_f(ld_prev(prevh + o), p);
            const float w1 = 1.f - w;
#pragma unroll
            for (int j = 0; j < 8; ++j) out[j] = fmaf(w, out[j], w1 * p[j]);
        }
    } else {
        float x0[8];
        h8_to_f(__ldg(x0h + o), x0);
        float v[8];
        if (slot >= 0) {
            const float4* vp = v32 + ((size_t)slot * kLPR + lane) * 2;
            const uint4 ua = ld_stream16(vp), ub = ld_stream16(vp + 1);
            v[0] = __uint_as_float(ua.x); v[1] = __uint_as_float(ua.y); v[2] = __uint_as_float(ua.z); v[3] = __uint_as_float(ua.w);
            v[4] = __uint_as_float(ub.x); v[5] = __uint_as_float(ub.y); v[6] = __uint_as_float(ub.z); v[7] = __uint_as_float(ub.w);
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float sc = __ldg(col_scale + lane * 8 + j);
            out[j] = t * (fmaf(alpha, acc[j], fmaf(sc, v[j], -x0[j])));
        }
    }
    const uint4 packed = f_to_h8(out);
    packed_out = packed;
    yh[o] = packed;
    // K5, direct form (long rows only): the same 16 bytes go into every peer GPU's copy of y.  The main kernel passes
    // no peers here and pushes its whole 4-KB row block at once (below)
#pragma unroll
    for (int i = 0; i < 7; ++i)
        if (i < peers.n) reinterpret_cast<uint4*>(peers.y[i])[o] = packed;
    h8_to_f(packed, out);
    if (MODE == 1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) out[j] = fabsf(out[j]);
    }
}

__device__ __forceinline__ void block_colsum_h(float (&v)[8], float* __restrict__ partial_row) {
    __shared__ float s_sum[kThreads / 32][kB];
#pragma unroll
    for (int off = kLPR; off < 32; off <<= 1)
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] += __shfl_xor_sync(0xffffffffu, v[j], off);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane < kLPR)
#pragma unroll
        for (int j = 0; j < 8; ++j) s_sum[warp][lane * 8 + j] = v[j];
    __syncthreads();
    if (threadIdx.x < kB) {
        float s = 0.f;
#pragma unroll
        for (int wi = 0; wi < kThreads / 32; ++wi) s += s_sum[wi][threadIdx.x];
        partial_row[threadIdx.x] = s;
    }
}

struct SweepArgs {
    int n_rows, row_base, long_thresh;
    const int* row_order;      // null = identity; else the local row handled by slot (cta * 64 + group): the 64 rows
                               // of a CTA sorted by length, so the 8 rows that share a warp finish together
    const int* row_ptr;
    const int2* cv;
    const uint4* xh;
    const int* slot_map;
    const uint4* rhs_h;
    const float4* v32;
    const float* col_scale;
    const uint4* prevh;
    uint4* yh;
    float alpha, w, t;
    float* partials;
};

// Single-GPU sweep: one block of 64 rows per CTA.  (Kept free of the exchange code of k_sweep_h_push below: sharing one
// body -- a block loop with the staging / bulk-copy code behind a uniform branch -- cost the plain sweep 13 %:
// 0.178 vs 0.157 ms on C3, profiles/r2_k1m_variants_d.txt.)
// 4 gathers in flight per lane at 6 CTAs per SM (8 / 4 and 6 / 5 measured slower, DESIGN.md section 4).
template <bool CHEB, int MODE, bool FINAL>
__global__ void __launch_bounds__(kThreads, 6)
k_sweep_h(const SweepArgs a) {
    constexpr int U = 4;
    const int g = threadIdx.x / kLPR, l = threadIdx.x % kLPR;
    const int slot_r = blockIdx.x * kGPB + g;
    float out[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) out[j] = 0.f;
    if (slot_r < a.n_rows) {
        const int r = a.row_order ? __ldg(a.row_order + slot_r) : slot_r;
        const int s = __ldg(a.row_ptr + r), e = __ldg(a.row_ptr + r + 1);
        if (e - s <= a.long_thresh) {
            float acc[8];
            uint4 packed;
            group_row_dot_h<U>(a.cv, s, e, a.xh + l, acc);
            row_epilogue_h<CHEB, MODE>(acc, a.row_base + r, l, a.slot_map, a.rhs_h, a.v32, a.col_scale, a.xh,
                                       a.prevh, a.yh, a.alpha, a.w, a.t, PeerOut(), out, packed);
        }
    }
    if (FINAL) block_colsum_h(out, a.partials + (size_t)blockIdx.x * kB);
}

// K5, the sharded sweep: the same row computation with the exchange fused in.
template <bool CHEB, int MODE, bool FINAL>
__global__ void __launch_bounds__(kThreads, 6)
k_sweep_h_push(const SweepArgs a, const PeerOut peers, const SweepSync sy) {
    constexpr int U = 4;
    // K5 staging: a block's 64 output rows are one contiguous 4-KB piece of y.  They are collected in shared memory and
    // pushed to every peer as ONE bulk copy per peer by the TMA engine (cp.async.bulk shared -> peer global over NVLink,
    // SASS UBLKCP): full-size NVLink packets, no store instructions on the SMs' LSUs, double-buffered so the copy of block
    // k overlaps the gathers of block k + 1.  Blocks that are not whole (ragged end, a long row inside) fall back to
    // coalesced 16-byte stores (thread t -> bytes [16 t, 16 t + 16)).
    __shared__ __align__(128) uint4 s_out[2][kThreads];
    __shared__ unsigned char s_valid[kGPB];
    sync_wait(sy);
    const int g = threadIdx.x / kLPR, l = threadIdx.x % kLPR;
    const bool push = peers.n > 0 && !(sy.debug & 2);    // uniform
    const int n_blocks = (a.n_rows + kGPB - 1) / kGPB;
    int buf = 0;
    // a persistent grid strides over the blocks, so the system-scope fence that must follow the peer writes (and waits
    // for their acknowledgements) is paid once per CTA at the end of the sweep, not once per 64 rows
    for (int blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
        const int slot_r = blk * kGPB + g;
        if (push) {
            // the bulk copies that read s_out[buf] two blocks ago must have finished reading it
            if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            if (l == 0) s_valid[g] = 0;
            __syncthreads();
        }
        float out[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) out[j] = 0.f;
        if (slot_r < a.n_rows) {
            const int r = a.row_order ? __ldg(a.row_order + slot_r) : slot_r;
            const int s = __ldg(a.row_ptr + r), e = __ldg(a.row_ptr + r + 1);
            if (e - s <= a.long_thresh) {
                float acc[8];
                uint4 packed;
                group_row_dot_h<U>(a.cv, s, e, a.xh + l, acc);
                row_epilogue_h<CHEB, MODE>(acc, a.row_base + r, l, a.slot_map, a.rhs_h, a.v32, a.col_scale, a.xh,
                                           a.prevh, a.yh, a.alpha, a.w, a.t, PeerOut(), out, packed);
                if (push) {
                    const int rl = r - blk * kGPB;       // row_order permutes rows inside their own 64-row block only
                    s_out[buf][rl * kLPR + l] = packed;
                    if (l == 0) s_valid[rl] = 1;
                }
            }
        }
        if (push) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the TMA engine
            const int whole = __syncthreads_and(s_valid[threadIdx.x / kLPR] != 0);
            const size_t o0 = (size_t)(a.row_base + blk * kGPB) * kLPR;
            if (whole && !(sy.debug & 4)) {
                if (threadIdx.x == 0) {
                    const uint32_t src = (uint32_t)__cvta_generic_to_shared(&s_out[buf][0]);
#pragma unroll
                    for (int i = 0; i < 7; ++i)
                        if (i < peers.n)
                            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                         ::"l"(reinterpret_cast<uint4*>(peers.y[i]) + o0), "r"(src), "r"((uint32_t)(kThreads * 16))
                                         : "memory");
                }
            } else if (s_valid[threadIdx.x / kLPR]) {
                const uint4 v = s_out[buf][threadIdx.x];
#pragma unroll
                for (int i = 0; i < 7; ++i)
                    if (i < peers.n) reinterpret_cast<uint4*>(peers.y[i])[o0 + threadIdx.x] = v;
            }
            if (threadIdx.x == 0) asm volatile("cp.async.bulk.commit_group;" ::: "memory");   // one group per block, empty or not
            buf ^= 1;
        }
        if (FINAL) {
            block_colsum_h(out, a.partials + (size_t)blk * kB);
            if (blk + (int)gridDim.x < n_blocks) __syncthreads();     // its shared scratch is reused by the next block
        }
    }
    if (push && threadIdx.x == 0) {
        if (sy.done_ctr != nullptr) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");      // all peer writes performed
        else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // staging buffers read; the kernel boundary orders the writes
    }
    sync_signal(sy);
}

__global__ void __launch_bounds__(kThreads)
k_sweep_long_segments_h(int n_seg, const int4* __restrict__ segs, const int2* __restrict__ cv,
                        const uint4* __restrict__ xh, float* __restrict__ seg_partial /* [n_seg, 32] */,
                        const SweepSync sy) {
    sync_wait(sy);
    constexpr int G = 32 / kLPR;
    const int warp = (blockIdx.x * kThreads + threadIdx.x) >> 5;
    if (warp >= n_seg) return;
    const int lane = threadIdx.x & 31;
    const int g = lane / kLPR, l = lane % kLPR;
    const int4 sg = __ldg(segs + warp);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int i = sg.y + g; i < sg.z; i += G) {
        const int2 c = __ldg(cv + i);
        fma8(acc, __int_as_float(c.y), __ldg(xh + (size_t)c.x * kLPR + l));
    }
#pragma unroll
    for (int off = kLPR; off < 32; off <<= 1)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], off);
    if (lane < kLPR)
#pragma unroll
        for (int j = 0; j < 8; ++j) seg_partial[(size_t)warp * kB + lane * 8 + j] = acc[j];
}

template <bool CHEB, int MODE, bool FINAL>
__global__ void __launch_bounds__(kThreads)
k_sweep_long_finalize_h(int n_long, const int* __restrict__ long_rows, const int* __restrict__ long_seg_ptr,
                        const float* __restrict__ seg_partial, const SweepArgs a, const PeerOut peers,
                        const SweepSync sy) {
    const int g = threadIdx.x / kLPR, l = threadIdx.x % kLPR;
    const int k = blockIdx.x * kGPB + g;
    float out[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) out[j] = 0.f;
    if (k < n_long) {
        const int r = __ldg(long_rows + k);
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.f;
        for (int s = __ldg(long_seg_ptr + k); s < __ldg(long_seg_ptr + k + 1); ++s)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] += seg_partial[(size_t)s * kB + l * 8 + j];
        uint4 packed;
        row_epilogue_h<CHEB, MODE>(acc, a.row_base + r, l, a.slot_map, a.rhs_h, a.v32, a.col_scale, a.xh, a.prevh,
                                   a.yh, a.alpha, a.w, a.t, peers, out, packed);
    }
    if (FINAL) block_colsum_h(out, a.partials + (size_t)blockIdx.x * kB);
    sync_signal(sy);
}

// stand-alone halves of the handshake, for the exchange points that are not sweeps (see api.cu)
__global__ void k_epoch_wait(const SweepSync sy) { sync_wait(sy); }
__global__ void k_epoch_signal(const SweepSync sy) { sync_signal(sy); }

// ---- dense prepare path (hrag_ppr: arbitrary reset vectors) ------------------------------------
// per-CTA column sums of a non-negative fp32 [N, 32] matrix -> partial[blockIdx, 32]
__global__ void __launch_bounds__(256)
k_colsum32_partial(const float* __restrict__ V, int64_t n_elems, float* __restrict__ partial) {
    float m = 0.f;                                   // thread's column = threadIdx.x % 32 (strides are multiples of 32)
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n_elems; i += (int64_t)gridDim.x * 256) m += V[i];
    __shared__ float s[256];
    s[threadIdx.x] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        for (int k = 1; k < 8; ++k) m += s[threadIdx.x + 32 * k];
        partial[(size_t)blockIdx.x * 32 + threadIdx.x] = m;
    }
}
// All entries of x = (I - aP)^-1 v are >= 0 and sum to <= sum(v) / (1 - a), so no entry of the
// scaled iterate can exceed fp16's range when  scale * sum(v) / (1 - a) <= 32768:
// scale[b] = 2^floor(log2(32768 (1 - a) / sum_b))      (sum == 0: an unused column -> 1)
__device__ __forceinline__ float column_scale(float sv, float one_minus_alpha) {
    return sv > 0.f ? exp2f(floorf(log2f(32768.f * one_minus_alpha / sv))) : 1.f;
}
__global__ void k_scales32(const double* __restrict__ vsum, float one_minus_alpha, float* __restrict__ scale) {
    scale[threadIdx.x] = column_scale((float)vsum[threadIdx.x], one_minus_alpha);
}
// V16[n, b] = fp16(scale[b] * V32[n, b])
__global__ void __launch_bounds__(256)
k_scale_to_half(const float4* __restrict__ V, int64_t n_vec8, const float* __restrict__ scale, uint4* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;       // one 8-column group
    if (i >= n_vec8) return;
    const int c0 = (int)(i & 3) * 8;
    const float4 a = __ldcs(V + 2 * i), b = __ldcs(V + 2 * i + 1);
    float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] *= __ldg(scale + c0 + j);
    out[i] = f_to_h8(f);
}

// ---- compact prepare path (stage B: passage weights + phrase seeds) ----------------------------
// Vc[p, b] = fp32(minmax(S[q0+b, p])) * fp32(pnw) for the P passage slots (HippoRAG.py:1626-1633; the
// product is formed in fp32 as numpy does for float32 * python float); columns b >= nb are 0.
// 32 passages x 32 queries per CTA through a shared-memory transpose: S is read along passages
// (coalesced), Vc written along queries.  partial[blockIdx, b] = the CTA's column sums.
__global__ void __launch_bounds__(256)
k_rhs_passages(int P, int nb, const float* __restrict__ S, int64_t ldS, int q0, const float2* __restrict__ minmax,
               float pnw, float* __restrict__ Vc, float* __restrict__ partial) {
    __shared__ float tile[32][33];
    __shared__ float red[8][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int p0 = blockIdx.x * 32;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int b = ty + 8 * k, p = p0 + tx;
        float v = 0.f;
        if (b < nb && p < P) {
            const float2 mm = __ldg(minmax + q0 + b);
            const float range = mm.y - mm.x;
            const float s = __ldcs(S + (size_t)(q0 + b) * ldS + p);
            const float nrm = range == 0.f ? 1.f : __fdiv_rn(s - mm.x, range);   // misc_utils.py:130-139
            v = nrm * pnw;
        }
        tile[b][tx] = v;
    }
    __syncthreads();
    float csum = 0.f;                                   // column tx over this thread's 4 passages
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int pl = ty + 8 * k;
        const float v = tile[tx][pl];
        if (p0 + pl < P) Vc[(size_t)(p0 + pl) * kB + tx] = v;
        csum += v;
    }
    red[ty][tx] = csum;
    __syncthreads();
    if (ty == 0) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += red[k][tx];
        partial[(size_t)blockIdx.x * kB + tx] = s;
    }
}

// One CTA: gives every distinct seed vertex of the sub-batch a slot (passage vertices keep theirs), adds the
// phrase weights (HippoRAG.py:1638 phrase + passage weights), finishes the column sums of v and derives the
// fp16 column scales.  Item i = (query b = i / slots_per_query, seed r = i % slots_per_query) owns slot P + i.
__global__ void __launch_bounds__(1024)
k_rhs_seeds(int P, int nb, int q0, int slots_per_query, const int* __restrict__ seed_vid,
            const float* __restrict__ seed_w, int* __restrict__ slot_map, int* __restrict__ slot_vid,
            float* __restrict__ Vc, const float* __restrict__ partial, int n_partial, float one_minus_alpha,
            double* __restrict__ vsum, float* __restrict__ scale) {
    __shared__ double s_sum[32][33];
    __shared__ double s_seed[32];
    const int t = threadIdx.x;
    if (t < 32) s_seed[t] = 0.0;
    __syncthreads();
    const int n_items = kB * slots_per_query;
    for (int i = t; i < n_items; i += 1024) {
        const int b = i / slots_per_query, r = i % slots_per_query;
        int created = -1;
        if (b < nb) {
            const int v = seed_vid[(size_t)(q0 + b) * slots_per_query + r];
            if (v >= 0) {
                const float w = seed_w[(size_t)(q0 + b) * slots_per_query + r];
                const int old = atomicCAS(slot_map + v, -1, P + i);
                const int slot = old < 0 ? P + i : old;
                if (old < 0) created = v;
                // (vertex, query) pairs are distinct; seed rows were zeroed by the caller, passage rows hold the
                // passage weight written by k_rhs_passages (stream order)
                atomicAdd(Vc + (size_t)slot * kB + b, w);
                atomicAdd(&s_seed[b], (double)w);
            }
        }
        slot_vid[P + i] = created;
    }
    const int col = t & 31, part = t >> 5;           // 32 columns x 32 partial lanes
    double acc = 0.0;
    for (int i = part; i < n_partial; i += 32) acc += (double)partial[(size_t)i * kB + col];
    s_sum[part][col] = acc;
    __syncthreads();
    if (t < 32) {
        double s = s_seed[t];
        for (int i = 0; i < 32; ++i) s += s_sum[i][t];
        vsum[t] = s;
        scale[t] = column_scale((float)s, one_minus_alpha);
    }
}

// rhs16[slot, :] = fp16(scale * Vc[slot, :]) for every slot, and the same row scattered into the dense
// first iterate x0 (zeroed by the caller): x0[vertex(slot), :]
__global__ void __launch_bounds__(256)
k_rhs_convert(int P, int n_slots, const int* __restrict__ passage_vid, const int* __restrict__ slot_vid,
              const float4* __restrict__ Vc, const float* __restrict__ scale, uint4* __restrict__ rhs16,
              uint4* __restrict__ x0) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;       // one 8-column group
    const int slot = (int)(i >> 2), l = (int)(i & 3);
    if (slot >= n_slots) return;
    const int vid = slot < P ? __ldg(passage_vid + slot) : __ldg(slot_vid + slot);
    const float4 a = __ldcs(Vc + 2 * i), b = __ldcs(Vc + 2 * i + 1);
    float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] *= __ldg(scale + l * 8 + j);
    const uint4 h = f_to_h8(f);
    rhs16[i] = h;
    if (vid >= 0) x0[(size_t)vid * kLPR + l] = h;
}

// undo k_rhs_seeds: seed vertices that were given a slot of their own go back to "no rhs"
__global__ void __launch_bounds__(1024)
k_slot_clear(int P, int nb, int q0, int slots_per_query, const int* __restrict__ seed_vid, int* __restrict__ slot_map) {
    const int n_items = kB * slots_per_query;
    for (int i = threadIdx.x; i < n_items; i += 1024) {
        const int b = i / slots_per_query, r = i % slots_per_query;
        if (b >= nb) continue;
        const int v = seed_vid[(size_t)(q0 + b) * slots_per_query + r];
        if (v >= 0 && slot_map[v] >= P) slot_map[v] = -1;
    }
}

__global__ void __launch_bounds__(256)
k_slot_map_init(int N, int* __restrict__ slot_map) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < N) slot_map[i] = -1;
}
__global__ void __launch_bounds__(256)
k_slot_map_passages(int P, const int* __restrict__ passage_vid, int* __restrict__ slot_map) {
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p < P) slot_map[passage_vid[p]] = p;
}

// relative L1 size of the refinement residual per column: rho[b] = (sum_i |r_i| / t) / (scale[b] * sum v);
// keeps the running maximum over every solve since the last reset (checked on the host, api.cu)
__global__ void k_residual_check(const double* __restrict__ rsum, const double* __restrict__ vsum,
                                 const float* __restrict__ scale, float inv_t, float* __restrict__ rho_max) {
    const int b = threadIdx.x;
    const double den = (double)scale[b] * vsum[b];
    float rho = den > 0.0 ? (float)(rsum[b] * (double)inv_t / den) : 0.f;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) rho = fmaxf(rho, __shfl_xor_sync(0xffffffffu, rho, off));
    if (b == 0 && rho > *rho_max) *rho_max = rho;
}

__global__ void __launch_bounds__(256)
k_gather_passage_scores_mixed(int P, int nb, int q0, const int* __restrict__ passage_vid,
                              const __half* __restrict__ X0, const __half* __restrict__ D, float inv_t,
                              const double* __restrict__ sum0, const double* __restrict__ sum1,
                              const int* __restrict__ mode, const float2* __restrict__ minmax, float* S, int64_t ldS) {
    const int64_t tI = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int p = (int)(tI / nb), b = (int)(tI % nb);
    if (p >= P) return;
    float* dst = S + (size_t)(q0 + b) * ldS + p;
    if (mode[q0 + b]) {
        const size_t o = (size_t)__ldg(passage_vid + p) * kB + b;
        const float z = __half2float(X0[o]) + inv_t * __half2float(D[o]);        // x = x0 + d
        const float tot = (float)(sum0[b] + (double)inv_t * sum1[b]);
        *dst = __fdiv_rn(z, tot);
    } else {
        const float2 mm = __ldg(minmax + q0 + b);
        const float range = mm.y - mm.x;
        *dst = range == 0.f ? 1.f : __fdiv_rn(*dst - mm.x, range);
    }
}

__global__ void __launch_bounds__(256)
k_state_to_scores_mixed(const __half* __restrict__ X0, const __half* __restrict__ D, float inv_t, int nb, int N,
                        const double* __restrict__ sum0, const double* __restrict__ sum1, float* __restrict__ out) {
    const int64_t tI = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int n = (int)(tI / nb), b = (int)(tI % nb);
    if (n >= N) return;
    const size_t o = (size_t)n * kB + b;
    const float z = __half2float(X0[o]) + inv_t * __half2float(D[o]);
    out[(size_t)b * N + n] = __fdiv_rn(z, (float)(sum0[b] + (double)inv_t * sum1[b]));
}

}  // namespace

int mixed_partial_rows(const PprGraph& g) {
    return (int)ceil_div(g.n_rows, kGPB) + (g.n_long ? (int)ceil_div(g.n_long, kGPB) : 0);
}

int epoch_wait(const SweepSync& sync, cudaStream_t st) {
    k_epoch_wait<<<1, 32, 0, st>>>(sync);
    count_launch();
    HRAG_CUDA(cudaGetLastError());
    return 0;
}
int epoch_signal(const SweepSync& sync, cudaStream_t st) {
    SweepSync sy = sync;
    sy.total_ctas = 1;
    k_epoch_signal<<<1, 32, 0, st>>>(sy);
    count_launch();
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

// One fp16 sweep (mode 0) or the residual sweep (mode 1) over the owned rows.
int mixed_sweep(const PprGraph& g, int mode, const void* xh, const int* slot_map, const void* rhs_h, const float* v32,
                const float* col_scale, const void* prevh, void* yh, float alpha, float w, float t, float* partials,
                int* n_partials, const PeerOut& peers, const SweepSync& sync, cudaStream_t st) {
    HRAG_CHECK(g.row_ptr && g.cv, "mixed_sweep: graph not loaded");
    const bool cheb = prevh != nullptr, fin = partials != nullptr;
    const int nb_rows = (int)ceil_div(g.n_rows, kGPB);
    const int nb_long = g.n_long ? (int)ceil_div(g.n_long, kGPB) : 0;
    SweepArgs a;
    a.n_rows = g.n_rows; a.row_base = g.row_lo; a.long_thresh = g.long_thresh;
    a.row_order = g.row_order;
    a.row_ptr = g.row_ptr; a.cv = g.cv;
    a.xh = reinterpret_cast<const uint4*>(xh);
    a.slot_map = slot_map;
    a.rhs_h = reinterpret_cast<const uint4*>(rhs_h);
    a.v32 = reinterpret_cast<const float4*>(v32);
    a.col_scale = col_scale;
    a.prevh = reinterpret_cast<const uint4*>(prevh);
    a.yh = reinterpret_cast<uint4*>(yh);
    a.alpha = alpha; a.w = w; a.t = t;
    a.partials = partials;
    SweepSync sy = sync;
    // sharded (fused exchange): a persistent grid, one system-scope fence per CTA (see k_sweep_h_push)
    static int persist_mult = -1;    // HRAG_MIXED_PERSIST=k: k x (6 CTAs per SM) persistent CTAs (default 1)
    if (persist_mult < 0) { const char* e = getenv("HRAG_MIXED_PERSIST"); persist_mult = e ? std::max(1, atoi(e)) : 1; }
    // HRAG_K5_MODE: 0 (default) = persistent grid, the epoch is published by the last CTA of the sweep itself (one system
    // fence per CTA, no extra launch; the staging ring is double-buffered so a block's bulk copies overlap the next
    // block's gathers); 1 = one CTA per 64-row block, no fence inside, the epoch is published by a one-warp kernel behind
    // the sweep (the kernel boundary orders the peer writes).  The wait is inside the sweep either way.  Measured
    // (profiles/r2_k5_*): equal on 2 GPUs (0.132 vs 0.135 ms), mode 0 ahead on 8 (0.124-0.130 vs 0.144 ms): without the
    // second staging buffer a CTA sits on its slot until the TMA engine has drained its 7 copies into a congested link.
    static int k5_mode = -1;
    if (k5_mode < 0) { const char* e = getenv("HRAG_K5_MODE"); k5_mode = e ? atoi(e) : 0; }
    const bool sharded = sync.flags != nullptr;
    const bool trailing_signal = sharded && k5_mode == 1;
    const int grid_rows = sharded && !trailing_signal ? std::min(nb_rows, g.num_sms * 6 * persist_mult) : nb_rows;
    sy.total_ctas = (unsigned)(grid_rows + nb_long);
    const SweepSync sy_full = sy;
    if (trailing_signal) sy.done_ctr = nullptr;          // the sweep kernels only wait
    SweepSync sy_wait_only = sy;
    sy_wait_only.done_ctr = nullptr;
    if (g.n_long) {
        k_sweep_long_segments_h<<<(unsigned)ceil_div((int64_t)g.n_seg * 32, kThreads), kThreads, 0, st>>>(
            g.n_seg, g.segs, g.cv, a.xh, g.seg_partial, sy_wait_only);
        count_launch();
    }
    SweepArgs al = a;
    al.partials = fin ? partials + (size_t)nb_rows * kB : nullptr;
#define HRAG_LAUNCH_H(C, M, F)                                                                                    \
    do {                                                                                                          \
        if (nb_rows) {                                                                                            \
            if (sharded) k_sweep_h_push<C, M, F><<<grid_rows, kThreads, 0, st>>>(a, peers, sy);                    \
            else k_sweep_h<C, M, F><<<grid_rows, kThreads, 0, st>>>(a);                                           \
            count_launch();                                                                                       \
        }                                                                                                         \
        if (nb_long) {                                                                                            \
            k_sweep_long_finalize_h<C, M, F><<<nb_long, kThreads, 0, st>>>(                                        \
                g.n_long, g.long_rows, g.long_seg_ptr, g.seg_partial, al, peers, sy);                             \
            count_launch();                                                                                       \
        }                                                                                                         \
    } while (0)
    if (mode == 1 && fin) HRAG_LAUNCH_H(false, 1, true);
    else if (mode == 1) HRAG_LAUNCH_H(false, 1, false);
    else if (cheb && fin) HRAG_LAUNCH_H(true, 0, true);
    else if (cheb) HRAG_LAUNCH_H(true, 0, false);
    else if (fin) HRAG_LAUNCH_H(false, 0, true);
    else HRAG_LAUNCH_H(false, 0, false);
#undef HRAG_LAUNCH_H
    if ((nb_rows + nb_long == 0 || trailing_signal) && sy.flags != nullptr) HRAG_TRY(epoch_signal(sy_full, st));
    if (n_partials) *n_partials = nb_rows + nb_long;
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

int mixed_prepare_rhs(const float* V32, int64_t n_rows, float alpha, float* partials, double* vsum, float* scale,
                      void* V16, cudaStream_t st) {
    const int64_t n_elems = n_rows * kB;
    const int nblk = (int)std::min<int64_t>(ceil_div(n_elems, 256), 1024);
    k_colsum32_partial<<<nblk, 256, 0, st>>>(V32, n_elems, partials);
    HRAG_TRY(colsum_reduce(partials, nblk, kB, vsum, st));
    k_scales32<<<1, kB, 0, st>>>(vsum, 1.f - alpha, scale);
    k_scale_to_half<<<(unsigned)ceil_div(n_elems / 8, 256), 256, 0, st>>>(reinterpret_cast<const float4*>(V32),
                                                                          n_elems / 8, scale,
                                                                          reinterpret_cast<uint4*>(V16));
    count_launch(3);
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

int slot_map_build(int N, int P, const int* passage_vid, int* slot_map, cudaStream_t st) {
    k_slot_map_init<<<(unsigned)ceil_div(N, 256), 256, 0, st>>>(N, slot_map);
    if (P) k_slot_map_passages<<<(unsigned)ceil_div(P, 256), 256, 0, st>>>(P, passage_vid, slot_map);
    count_launch(2);
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

int compact_rhs_partial_rows(int P) { return (int)ceil_div(std::max(P, 1), 32); }

int compact_prepare_rhs(const SeedTables& t, int nb, int q0, const float* S, int64_t ldS, const float2* minmax,
                        float pnw, int slots_per_query, const int* seed_vid, const float* seed_w, float alpha,
                        int* slot_map, int* slot_vid, float* Vc, void* rhs16, void* x0_dense, int64_t n_nodes,
                        float* partials, double* vsum, float* scale, cudaStream_t st) {
    const int P = t.n_passages;
    const int n_seed_slots = kB * slots_per_query;
    HRAG_CHECK(slots_per_query > 0, "compact_prepare_rhs: slots_per_query must be positive");
    const int nblk = compact_rhs_partial_rows(P);
    HRAG_CUDA(cudaMemsetAsync(x0_dense, 0, (size_t)n_nodes * kB * 2, st));
    HRAG_CUDA(cudaMemsetAsync(Vc + (size_t)P * kB, 0, (size_t)n_seed_slots * kB * sizeof(float), st));
    k_rhs_passages<<<nblk, 256, 0, st>>>(P, nb, S, ldS, q0, minmax, pnw, Vc, partials);
    k_rhs_seeds<<<1, 1024, 0, st>>>(P, nb, q0, slots_per_query, seed_vid, seed_w, slot_map, slot_vid, Vc,
                                            partials, nblk, 1.f - alpha, vsum, scale);
    const int n_slots = P + n_seed_slots;
    k_rhs_convert<<<(unsigned)ceil_div((int64_t)n_slots * kLPR, 256), 256, 0, st>>>(
        P, n_slots, t.passage_vid, slot_vid, reinterpret_cast<const float4*>(Vc), scale,
        reinterpret_cast<uint4*>(rhs16), reinterpret_cast<uint4*>(x0_dense));
    count_launch(3);
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

int compact_release_slots(int P, int nb, int q0, int slots_per_query, const int* seed_vid, int* slot_map,
                          cudaStream_t st) {
    k_slot_clear<<<1, 1024, 0, st>>>(P, nb, q0, slots_per_query, seed_vid, slot_map);
    count_launch();
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

int residual_check(const double* rsum, const double* vsum, const float* scale, float inv_t, float* rho_max,
                   cudaStream_t st) {
    k_residual_check<<<1, kB, 0, st>>>(rsum, vsum, scale, inv_t, rho_max);
    count_launch();
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

int gather_passage_scores_mixed(const SeedTables& t, int nb, int q0, const void* X0, const void* D, float inv_t,
                                const double* sum0, const double* sum1, const int* mode, const float2* minmax,
                                float* S, int64_t ldS, cudaStream_t st) {
    if (t.n_passages == 0 || nb == 0) return 0;
    const int64_t total = (int64_t)t.n_passages * nb;
    k_gather_passage_scores_mixed<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(
        t.n_passages, nb, q0, t.passage_vid, reinterpret_cast<const __half*>(X0), reinterpret_cast<const __half*>(D),
        inv_t, sum0, sum1, mode, minmax, S, ldS);
    count_launch();
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

int state_to_scores_mixed(const void* X0, const void* D, float inv_t, int nb, int N, const double* sum0,
                          const double* sum1, float* out, cudaStream_t st) {
    const int64_t total = (int64_t)N * nb;
    k_state_to_scores_mixed<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(
        reinterpret_cast<const __half*>(X0), reinterpret_cast<const __half*>(D), inv_t, nb, N, sum0, sum1, out);
    count_launch();
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace hrag
