// Launchers of the hand-written sm_100a kernels (K1..K4).  Host-callable C++; the C ABI in
// api.cu composes them.  All pointers are device pointers; all launches go to `stream`.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace hrag {

struct SeedTables;

// ----------------------------------------------------------------------------- K1: PPR SpMM
// CSR of P = W D^-1 for the rows this GPU owns, packed as (col, val) pairs.
struct PprGraph {
    int n_global = 0;        // N
    int row_lo = 0;          // first global row owned
    int n_rows = 0;          // rows owned
    int64_t nnz = 0;
    int* row_ptr = nullptr;  // [n_rows + 1]
    int2* cv = nullptr;      // [nnz]  {col, __float_as_int(val)}
    // rows longer than `long_thresh` are split into warp-sized segments
    int long_thresh = 0;
    int n_long = 0;
    int* long_rows = nullptr;     // [n_long] local row ids
    int* long_seg_ptr = nullptr;  // [n_long + 1] offsets into segs
    int n_seg = 0;
    int4* segs = nullptr;         // [n_seg] {local row, begin, end, 0}
    float* seg_partial = nullptr; // [n_seg * Bmax]
    int max_batch = 0;
    int num_sms = 148;
    int* row_order = nullptr;     // [n_rows] fp16 sweep: rows of each 64-row CTA block sorted by length (desc)
};

// One sweep  y[i,:] = w * (alpha * sum_j P[i,j] x[j,:] + v[i,:]) + (1 - w) * prev[i,:]
// over the owned rows.  x, v, prev, y are [N, B] row-major fp32 (global row indexing);
// prev may be null (w == 1) and may alias y.  If colsum_partials != null the per-block
// column sums of y are written there ([n_blocks_total, B] floats) and *n_partials gets the
// row count.  B in {4, 8, 16, 32, 64}.
int ppr_sweep(const PprGraph& g, int B, const float* x, const float* v, const float* prev, float* y,
              float alpha, float w, float* colsum_partials, int* n_partials, cudaStream_t stream);
int ppr_sweep_partial_rows(const PprGraph& g, int B);  // rows of colsum_partials a sweep writes

// ---- K5: fused sweep + exchange for node-range sharding ------------------------------------------
// The sweep's epilogue stores each output row into the same offset of every peer GPU's buffer
// (IPC-mapped over NVLink); epochs published through flag words replace the per-sweep all-gather.
struct PeerOut {
    void* y[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // peers' copy of this sweep's y
    int n = 0;
};
// Epoch handshake of the fused exchange, carried by the sweep kernels themselves: every CTA waits until all
// peers' flag words reach `need`; the last CTA to finish publishes `epoch` into the peers' flag word of this rank.
struct SweepSync {
    const unsigned long long* flags = nullptr;   // local flag words, one per rank (null = single GPU / NCCL path)
    unsigned long long need = 0;
    int world = 1, rank = 0;
    int* error_flag = nullptr;                   // set when a peer never showed up (bounded spin)
    unsigned int* done_ctr = nullptr;            // CTAs finished in this sweep (self-resetting); null = wait only
    unsigned int total_ctas = 0;                 // filled in by mixed_sweep
    unsigned long long* remote[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int n_remote = 0;
    unsigned long long epoch = 0;
    int debug = 0;            // profiling only (hrag_set_tuning k5_debug): 1 = no system fence, 2 = no peer writes, 4 = LSU stores, not TMA
};

// ---- mixed-precision solver (ppr_mixed.cu): fp16 state [N, 32], fp32 arithmetic ------------
// mode 0: yh = w * (alpha * P xh + rhs) + (1 - w) * prevh ;  mode 1 (residual):
// yh = t * (col_scale * v32 - xh + alpha * P xh), partials (if given) = column sums of |yh|.
// rhs_h / v32 are [n_slots, 32] arrays addressed through slot_map[node] (-1 = zero row); slot_map == null
// means dense [N, 32].  partials as in ppr_sweep ([rows, 32] floats).
int mixed_sweep(const PprGraph& g, int mode, const void* xh, const int* slot_map, const void* rhs_h,
                const float* v32, const float* col_scale, const void* prevh, void* yh, float alpha, float w,
                float t, float* partials, int* n_partials, const PeerOut& peers, const SweepSync& sync,
                cudaStream_t stream);
int mixed_partial_rows(const PprGraph& g);
// vsum[32] <- column sums of V32 [n_rows, 32] (>= 0; `partials` = scratch of >= 1024*32 floats);
// scale[b] = 2^floor(log2(32768 (1 - alpha) / vsum[b])) -- overflow-proof, see ppr_mixed.cu;
// V16 = fp16(scale * V32).
int mixed_prepare_rhs(const float* V32, int64_t n_rows, float alpha, float* partials, double* vsum, float* scale,
                      void* V16, cudaStream_t stream);
// Compact right-hand side of stage B (reset vector of graph_search_with_fact_entities): slot_map[passage_vid[p]] = p,
// everything else -1.
int slot_map_build(int N, int P, const int* passage_vid, int* slot_map, cudaStream_t stream);
int compact_rhs_partial_rows(int P);
// Builds, for the nb queries [q0, q0 + nb) of a chunk: Vc [P + 32*slots_per_query, 32] fp32 (passage weights
// pnw * minmax(S) on the passage slots, phrase weights on freshly assigned seed slots), its column sums / fp16
// scales, rhs16 = fp16(scale * Vc), and the dense first iterate x0_dense [n_nodes, 32] fp16.
int compact_prepare_rhs(const SeedTables& t, int nb, int q0, const float* S, int64_t ldS, const float2* minmax,
                        float pnw, int slots_per_query, const int* seed_vid, const float* seed_w, float alpha,
                        int* slot_map, int* slot_vid, float* Vc, void* rhs16, void* x0_dense, int64_t n_nodes,
                        float* partials, double* vsum, float* scale, cudaStream_t stream);
int compact_release_slots(int P, int nb, int q0, int slots_per_query, const int* seed_vid, int* slot_map,
                          cudaStream_t stream);
// rho_max = max(rho_max, max_b (rsum[b] / t) / (scale[b] * vsum[b])): relative L1 residual of the iterate
int residual_check(const double* rsum, const double* vsum, const float* scale, float inv_t, float* rho_max,
                   cudaStream_t stream);
int epoch_wait(const SweepSync& sync, cudaStream_t stream);
int epoch_signal(const SweepSync& sync, cudaStream_t stream);
int gather_passage_scores_mixed(const SeedTables& t, int nb, int q0, const void* X0, const void* D, float inv_t,
                                const double* sum0, const double* sum1, const int* mode, const float2* minmax,
                                float* S, int64_t ldS, cudaStream_t stream);
int state_to_scores_mixed(const void* X0, const void* D, float inv_t, int nb, int N, const double* sum0,
                          const double* sum1, float* out, cudaStream_t stream);

// sums[b] = sum over rows of partials[r, b], accumulated in fp64.
int colsum_reduce(const float* partials, int n_partials, int B, double* sums, cudaStream_t stream);

// ----------------------------------------------------------------------------- K2: similarity
// S[b, m] = <Q[b, :], E[m, :]>  (fp32 FMA).  Q [Bq, dim], E [M, dim], S [Bq, ldS].
int sim_fp32(const float* Q, int Bq, const float* E, int64_t M, int dim, float* S, int64_t ldS,
             cudaStream_t stream);

// Tensor-core variant (sim_tc.cu): operands pre-split into bf16 hi/lo ([rows, dim] each,
// x = hi + lo); n_seg = 4 -> all four hi/lo products (fp32-faithful), n_seg = 1 -> q_hi.e_hi only.
// dim % 8 == 0, ldS % 4 == 0.
int split_bf16(const float* x, int64_t n, void* hi, void* lo, cudaStream_t stream);
// With part_mm / part_keys != null the epilogue is FUSED: no score matrix is written; per
// (query, 256-column tile) it emits min/max (part_mm [Bq, n_tiles]) and the 8 best rank keys
// (part_keys [Bq, n_tiles, 8]); merge_minmax_topk() finishes the selection.
int sim_tc(const void* q_hi, const void* q_lo, int Bq, const void* e_hi, const void* e_lo, int64_t M, int dim,
           int n_seg, float* S, int64_t ldS, float2* part_mm, uint64_t* part_keys, int num_sms,
           cudaStream_t stream);
int sim_tc_n_tiles(int64_t M);
// Threshold epilogue (index-time synonymy KNN, SURVEY.md 8(f)-2): no score matrix; every score >= thr is appended as
// a rank key to cand_keys[query, :cand_cap] and counted in cand_count[query] (zeroed by the caller; it keeps counting
// past cand_cap).  sort_candidates then orders each list and emits the first kmax (cap must be kCandidateCap).
constexpr int kCandidateCap = 512;
int sim_tc_threshold(const void* q_hi, const void* q_lo, int Bq, const void* e_hi, const void* e_lo, int64_t M, int dim,
                     int n_seg, float thr, uint64_t* cand_keys, int* cand_count, int cand_cap, int num_sms,
                     cudaStream_t stream);
int sort_candidates(const uint64_t* cand_keys, const int* cand_count, int rows, int cap, int kmax, int* out_ids,
                    float* out_scores, int* n_found, cudaStream_t stream);
int merge_minmax_topk(const float2* part_mm, const uint64_t* part_keys, int rows, int n_tiles, int64_t M, int k,
                      float2* minmax, int* top_idx, float* top_score, int* n_valid, cudaStream_t stream);
// Strided form (entry of (row, tile) at row * row_stride + tile * tile_stride) with an index offset; raw_keys != null
// writes the k best keys of each row unnormalised ([rows, k], 0 = none) instead of idx / score -- the local half of a
// fact-sharded stage A, whose per-rank results the same kernel merges after the all-gather.
int merge_minmax_topk_ex(const float2* part_mm, const uint64_t* part_keys, int rows, int n_tiles, int64_t row_stride,
                         int64_t tile_stride, int64_t idx_offset, int64_t M, int k, float2* minmax, int* top_idx,
                         float* top_score, int* n_valid, uint64_t* raw_keys, cudaStream_t stream);

// ----------------------------------------------------------------------------- selection
// Per row of S [rows, ld] (first M columns): min, max -> minmax[row] = {min, max}; if k > 0
// also the k best (score desc, index asc) -> top_idx[row, k], top_score[row, k] min-max
// normalised (all-equal -> 1), n_valid[row] = min(k, M).  k <= 8.
int row_minmax_topk(const float* S, int rows, int64_t M, int64_t ld, int k, float2* minmax,
                    int* top_idx, float* top_score, int* n_valid, cudaStream_t stream);

// scores[row, j] (raw, from row_topk) <- min-max normalised with minmax[row]; n_valid[row] = min(k, M)
int topk_normalize(int rows, int k, int64_t M, const float2* minmax, const int* ids, float* scores, int* n_valid,
                   cudaStream_t stream);

// In place: S[row, :M] <- min-max normalised with minmax[row] (all-equal -> 1).
int minmax_apply(float* S, int rows, int64_t M, int64_t ld, const float2* minmax, cudaStream_t stream);

// Per row of S [rows, ld]: the k (<= 2048) best of the first M columns by (score desc,
// index asc), sorted.  out_ids / out_scores are [rows, k]; missing entries (k > M) = -1 / 0.
int row_topk(const float* S, int rows, int64_t M, int64_t ld, int k, int* out_ids, float* out_scores,
             cudaStream_t stream);

// ----------------------------------------------------------------------------- K3: seeds
constexpr int kMaxKeptFacts = 32;                       // kept facts per query (linking_top_k, config_utils.py:184)
constexpr int kSeedSlotsPerQuery = 2 * kMaxKeptFacts;   // subject + object of every kept fact
struct SeedTables {
    int n_nodes = 0;
    int n_passages = 0;
    int64_t n_facts = 0;
    int* passage_vid = nullptr;
    int* fact_subj_vid = nullptr;
    int* fact_obj_vid = nullptr;
    int* ent_chunk_count = nullptr;
};

// V[passage_vid[p], b] = pnw * minmax(S[q0 + b, p]) for b < nb (V is [N, B], zeroed first by
// the caller; columns b >= nb stay zero).
int seed_passages(const SeedTables& t, int B, int nb, const float* S, int64_t ldS, int q0,
                  const float2* minmax, float pnw, float* V, cudaStream_t stream);
// Phrase seeds of graph_search_with_fact_entities for the nq queries of a chunk: the kept facts'
// subject/object vertices get mean(score / chunk_count), the link_top_k best survive ->
// seed_vid / seed_w [nq, kSeedSlotsPerQuery] (-1 = unused); mode[q] = 1 (PPR) or 0 (DPR fallback: no kept fact / flagged).
int seed_entities(const SeedTables& t, int nq, const int* kept_idx, const float* kept_score, int k_facts,
                  const uint8_t* dpr_only, int link_top_k, int* seed_vid, float* seed_w, int* mode,
                  cudaStream_t stream);
// V[seed_vid[q0 + b, :], b] += seed_w[q0 + b, :] for b < nb.
int seed_scatter(int B, int nb, int q0, const int* seed_vid, const float* seed_w, float* V, cudaStream_t stream);

// ----------------------------------------------------------------------------- K4: gather
// PPR rows: S[q0 + b, p] = Z[passage_vid[p], b] / sums[b]; DPR-fallback rows (mode == 0):
// S[q0 + b, p] = minmax(S[q0 + b, p]) in place.
int gather_passage_scores(const SeedTables& t, int B, int nb, int q0, const float* Z, const double* sums,
                          const int* mode, const float2* minmax, float* S, int64_t ldS,
                          cudaStream_t stream);

// Sanitise + transpose host-layout reset vectors: V[n, b] = max(R[b, n], 0) (NaN -> 0).
int reset_to_state(const float* R, int nb, int N, int B, float* V, cudaStream_t stream);
// out[b, n] = Z[n, b] / sums[b]
int state_to_scores(const float* Z, int nb, int N, int B, const double* sums, float* out, cudaStream_t stream);

void count_launch(int n = 1);
int64_t launches_since_reset();
void reset_launch_counter();

}  // namespace hrag
