// K1 -- batched CSR SpMM sweep of the Personalized-PageRank iteration (sm_100a).
//
// Replaces the numeric core of HippoRAG.run_ppr (reference HippoRAG.py:1736-1743, which
// hands one reset vector at a time to igraph/PRPACK) with a batched fixed-point sweep
//     y[i,:] = w * (alpha * sum_j P[i,j] x[j,:] + v[i,:]) + (1 - w) * prev[i,:]
// over B right-hand sides at once.  w == 1 is the plain Neumann/power sweep
// z <- alpha P z + v; w != 1 is one Chebyshev semi-iteration step on the same fixed point.
// The L1 normalisation of the result (pi = z / sum z) needs only the column sums of the
// last iterate, which the last sweep's epilogue produces with warp-level reductions.
//
// Data layout: state matrices are [N, B] row-major fp32 (node-major, batch contiguous), so
// the gather of x[j,:] for a non-zero (i, j) is one contiguous 4B-byte segment (>= one
// 32-byte sector for B >= 8) and a group of B/4 lanes moves it with one 16-byte load per
// lane.  The matrix is CSR with (col, val) packed in 8 bytes so one load fetches both.
//
// Mapping: a group of LPR = B/4 lanes owns one row; 256/LPR rows per CTA; the row's
// non-zeros are walked four at a time so four independent gathers are in flight per lane
// (the sweep is bound by gather latency x bandwidth, not by FMA issue).  Rows longer than
// `long_thresh` are cut into segments handled one warp each (all groups of the warp stride
// through the segment, shuffle-reduce), then summed in a fixed order by a finalize kernel:
// deterministic, no atomics, no tail from a 10^5-degree hub.
//
// Roofline (DESIGN.md): HBM-bound; algorithmic bytes per sweep =
//     nnz * 8 + (n_rows + 1) * 4 + 3 * n_rows * B * 4.
#include "common.cuh"
#include "kernels.h"

namespace hrag {

static int64_t g_launches = 0;
int64_t launches_since_reset() { return g_launches; }
void reset_launch_counter() { g_launches = 0; }
void count_launch(int n) { g_launches += n; }

namespace {

constexpr int kThreads = 256;

template <int LPR>
__device__ __forceinline__ float4 group_row_dot(const int2* __restrict__ cv, int s, int e,
                                                const float4* __restrict__ x4 /* already + lane */) {
    float4 acc = f4_zero();
    int i = s;
    for (; i + 4 <= e; i += 4) {
        const int2 c0 = __ldg(cv + i), c1 = __ldg(cv + i + 1), c2 = __ldg(cv + i + 2), c3 = __ldg(cv + i + 3);
        const float4 a0 = __ldg(x4 + (size_t)c0.x * LPR);
        const float4 a1 = __ldg(x4 + (size_t)c1.x * LPR);
        const float4 a2 = __ldg(x4 + (size_t)c2.x * LPR);
        const float4 a3 = __ldg(x4 + (size_t)c3.x * LPR);
        f4_fma(acc, __int_as_float(c0.y), a0);
        f4_fma(acc, __int_as_float(c1.y), a1);
        f4_fma(acc, __int_as_float(c2.y), a2);
        f4_fma(acc, __int_as_float(c3.y), a3);
    }
    for (; i < e; ++i) {
        const int2 c = __ldg(cv + i);
        f4_fma(acc, __int_as_float(c.y), __ldg(x4 + (size_t)c.x * LPR));
    }
    return acc;
}

template <int LPR, bool CHEB>
__device__ __forceinline__ float4 row_epilogue(float4 acc, size_t o, const float4* __restrict__ v4,
                                               const float4* prev4, float4* y4, float alpha, float w) {
    const float4 vv = ld_stream_f4(v4 + o);
    float4 out;
    out.x = fmaf(alpha, acc.x, vv.x);
    out.y = fmaf(alpha, acc.y, vv.y);
    out.z = fmaf(alpha, acc.z, vv.z);
    out.w = fmaf(alpha, acc.w, vv.w);
    if (CHEB) {
        const float4 p = prev4[o];
        const float w1 = 1.f - w;
        out.x = fmaf(w, out.x, w1 * p.x);
        out.y = fmaf(w, out.y, w1 * p.y);
        out.z = fmaf(w, out.z, w1 * p.z);
        out.w = fmaf(w, out.w, w1 * p.w);
    }
    y4[o] = out;
    return out;
}

// Column sums of the per-thread float4 `out` over the whole CTA -> partial[blockIdx, B].
template <int LPR>
__device__ __forceinline__ void block_colsum(float4 out, float* __restrict__ partial_row) {
    constexpr int B = LPR * 4;
    __shared__ float s_sum[kThreads / 32][B];
#pragma unroll
    for (int off = LPR; off < 32; off <<= 1) {
        out.x += __shfl_xor_sync(0xffffffffu, out.x, off);
        out.y += __shfl_xor_sync(0xffffffffu, out.y, off);
        out.z += __shfl_xor_sync(0xffffffffu, out.z, off);
        out.w += __shfl_xor_sync(0xffffffffu, out.w, off);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane < LPR && lane < 32) {
        s_sum[warp][lane * 4 + 0] = out.x;
        s_sum[warp][lane * 4 + 1] = out.y;
        s_sum[warp][lane * 4 + 2] = out.z;
        s_sum[warp][lane * 4 + 3] = out.w;
    }
    __syncthreads();
    if (threadIdx.x < B) {
        float s = 0.f;
#pragma unroll
        for (int wi = 0; wi < kThreads / 32; ++wi) s += s_sum[wi][threadIdx.x];
        partial_row[threadIdx.x] = s;
    }
}

// ---- short rows: one group of LPR lanes per row ------------------------------------------
template <int LPR, bool CHEB, bool FINAL>
__global__ void __launch_bounds__(kThreads, 6)
k_sweep_rows(int n_rows, int row_base, int long_thresh, const int* __restrict__ row_ptr,
             const int2* __restrict__ cv, const float4* __restrict__ x4, const float4* __restrict__ v4,
             const float4* prev4, float4* y4, float alpha, float w, float* __restrict__ partials) {
    constexpr int GPB = kThreads / LPR;
    const int g = threadIdx.x / LPR, l = threadIdx.x % LPR;
    const int r = blockIdx.x * GPB + g;
    float4 out = f4_zero();
    if (r < n_rows) {
        const int s = __ldg(row_ptr + r), e = __ldg(row_ptr + r + 1);
        if (e - s <= long_thresh) {
            const float4 acc = group_row_dot<LPR>(cv, s, e, x4 + l);
            out = row_epilogue<LPR, CHEB>(acc, (size_t)(row_base + r) * LPR + l, v4, prev4, y4, alpha, w);
        }
    }
    if (FINAL) block_colsum<LPR>(out, partials + (size_t)blockIdx.x * (LPR * 4));
}

// ---- long rows: one warp per segment, groups stride through it ----------------------------
template <int LPR>
__global__ void __launch_bounds__(kThreads)
k_sweep_long_segments(int n_seg, const int4* __restrict__ segs, const int2* __restrict__ cv,
                      const float4* __restrict__ x4, float4* __restrict__ seg_partial4) {
    constexpr int G = 32 / LPR;  // groups per warp
    const int warp = (blockIdx.x * kThreads + threadIdx.x) >> 5;
    if (warp >= n_seg) return;
    const int lane = threadIdx.x & 31;
    const int g = lane / LPR, l = lane % LPR;
    const int4 sg = __ldg(segs + warp);
    float4 acc = f4_zero();
    int i = sg.y + g;
    for (; i + 3 * G < sg.z; i += 4 * G) {
        const int2 c0 = __ldg(cv + i), c1 = __ldg(cv + i + G), c2 = __ldg(cv + i + 2 * G), c3 = __ldg(cv + i + 3 * G);
        const float4 a0 = __ldg(x4 + (size_t)c0.x * LPR + l);
        const float4 a1 = __ldg(x4 + (size_t)c1.x * LPR + l);
        const float4 a2 = __ldg(x4 + (size_t)c2.x * LPR + l);
        const float4 a3 = __ldg(x4 + (size_t)c3.x * LPR + l);
        f4_fma(acc, __int_as_float(c0.y), a0);
        f4_fma(acc, __int_as_float(c1.y), a1);
        f4_fma(acc, __int_as_float(c2.y), a2);
        f4_fma(acc, __int_as_float(c3.y), a3);
    }
    for (; i < sg.z; i += G) {
        const int2 c = __ldg(cv + i);
        f4_fma(acc, __int_as_float(c.y), __ldg(x4 + (size_t)c.x * LPR + l));
    }
#pragma unroll
    for (int off = LPR; off < 32; off <<= 1) {
        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, off);
        acc.y += __shfl_xor_sync(0xffffffffu, acc.y, off);
        acc.z += __shfl_xor_sync(0xffffffffu, acc.z, off);
        acc.w += __shfl_xor_sync(0xffffffffu, acc.w, off);
    }
    if (lane < LPR) seg_partial4[(size_t)warp * LPR + lane] = acc;
}

template <int LPR, bool CHEB, bool FINAL>
__global__ void __launch_bounds__(kThreads)
k_sweep_long_finalize(int n_long, int row_base, const int* __restrict__ long_rows,
                      const int* __restrict__ long_seg_ptr, const float4* __restrict__ seg_partial4,
                      const float4* __restrict__ v4, const float4* prev4, float4* y4, float alpha, float w,
                      float* __restrict__ partials) {
    constexpr int GPB = kThreads / LPR;
    const int g = threadIdx.x / LPR, l = threadIdx.x % LPR;
    const int k = blockIdx.x * GPB + g;
    float4 out = f4_zero();
    if (k < n_long) {
        const int r = __ldg(long_rows + k);
        float4 acc = f4_zero();
        for (int s = __ldg(long_seg_ptr + k); s < __ldg(long_seg_ptr + k + 1); ++s)
            f4_add(acc, seg_partial4[(size_t)s * LPR + l]);
        out = row_epilogue<LPR, CHEB>(acc, (size_t)(row_base + r) * LPR + l, v4, prev4, y4, alpha, w);
    }
    if (FINAL) block_colsum<LPR>(out, partials + (size_t)blockIdx.x * (LPR * 4));
}

__global__ void __launch_bounds__(256)
k_colsum_reduce(const float* __restrict__ partials, int n_partials, int B, double* __restrict__ sums) {
    // one CTA per column; fp64 accumulation (an fp32 running sum over 10^4 partials costs ~1e-6)
    __shared__ double s[256];
    const int b = blockIdx.x;
    double acc = 0.0;
    for (int r = threadIdx.x; r < n_partials; r += 256) acc += (double)partials[(size_t)r * B + b];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if (threadIdx.x < off) s[threadIdx.x] += s[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) sums[b] = s[0];
}

template <int LPR>
int launch_sweep(const PprGraph& g, const float* x, const float* v, const float* prev, float* y, float alpha,
                 float w, float* partials, int* n_partials, cudaStream_t st) {
    constexpr int GPB = kThreads / LPR;
    const bool cheb = prev != nullptr;
    const bool fin = partials != nullptr;
    const int nb_rows = (int)ceil_div(g.n_rows, GPB);
    const int nb_long = g.n_long ? (int)ceil_div(g.n_long, GPB) : 0;
    const float4* x4 = reinterpret_cast<const float4*>(x);
    const float4* v4 = reinterpret_cast<const float4*>(v);
    const float4* p4 = reinterpret_cast<const float4*>(prev);
    float4* y4 = reinterpret_cast<float4*>(y);
    if (g.n_long) {
        k_sweep_long_segments<LPR><<<(unsigned)ceil_div((int64_t)g.n_seg * 32, kThreads), kThreads, 0, st>>>(
            g.n_seg, g.segs, g.cv, x4, reinterpret_cast<float4*>(g.seg_partial));
        count_launch();
    }
    float* part_long = fin ? partials + (size_t)nb_rows * LPR * 4 : nullptr;
#define HRAG_LAUNCH(C, F)                                                                              \
    do {                                                                                               \
        if (nb_rows) {                                                                                 \
            k_sweep_rows<LPR, C, F><<<nb_rows, kThreads, 0, st>>>(g.n_rows, g.row_lo, g.long_thresh,   \
                                                                  g.row_ptr, g.cv, x4, v4, p4, y4,     \
                                                                  alpha, w, partials);                 \
            count_launch();                                                                            \
        }                                                                                              \
        if (nb_long) {                                                                                 \
            k_sweep_long_finalize<LPR, C, F><<<nb_long, kThreads, 0, st>>>(                            \
                g.n_long, g.row_lo, g.long_rows, g.long_seg_ptr,                                       \
                reinterpret_cast<const float4*>(g.seg_partial), v4, p4, y4, alpha, w, part_long);      \
            count_launch();                                                                            \
        }                                                                                              \
    } while (0)
    if (cheb && fin) HRAG_LAUNCH(true, true);
    else if (cheb) HRAG_LAUNCH(true, false);
    else if (fin) HRAG_LAUNCH(false, true);
    else HRAG_LAUNCH(false, false);
#undef HRAG_LAUNCH
    if (n_partials) *n_partials = nb_rows + nb_long;
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace

int ppr_sweep_partial_rows(const PprGraph& g, int B) {
    const int GPB = kThreads / (B / 4);
    return (int)ceil_div(g.n_rows, GPB) + (g.n_long ? (int)ceil_div(g.n_long, GPB) : 0);
}

int ppr_sweep(const PprGraph& g, int B, const float* x, const float* v, const float* prev, float* y,
              float alpha, float w, float* colsum_partials, int* n_partials, cudaStream_t stream) {
    HRAG_CHECK(g.row_ptr && g.cv, "ppr_sweep: graph not loaded");
    HRAG_CHECK(B <= g.max_batch, "ppr_sweep: batch wider than the graph was prepared for");
    switch (B) {
        case 4:  return launch_sweep<1>(g, x, v, prev, y, alpha, w, colsum_partials, n_partials, stream);
        case 8:  return launch_sweep<2>(g, x, v, prev, y, alpha, w, colsum_partials, n_partials, stream);
        case 16: return launch_sweep<4>(g, x, v, prev, y, alpha, w, colsum_partials, n_partials, stream);
        case 32: return launch_sweep<8>(g, x, v, prev, y, alpha, w, colsum_partials, n_partials, stream);
        case 64: return launch_sweep<16>(g, x, v, prev, y, alpha, w, colsum_partials, n_partials, stream);
        default: break;
    }
    set_error("ppr_sweep: batch width must be one of 4, 8, 16, 32, 64");
    return 2;
}

int colsum_reduce(const float* partials, int n_partials, int B, double* sums, cudaStream_t stream) {
    k_colsum_reduce<<<B, 256, 0, stream>>>(partials, n_partials, B, sums);
    count_launch();
    HRAG_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace hrag
