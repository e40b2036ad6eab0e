/* hrag_b200.h -- C ABI of libhrag_b200.so: HippoRAG's online retrieval hot path on B200 (sm_100a).
 *
 * The reference (OSU-NLP-Group/HippoRAG) is pure Python and has no FFI of its own; the
 * boundary this library replaces is a set of methods on the `HippoRAG` object.  Each entry
 * point below names the reference code it stands in for (paths under
 * /root/reference/src/hipporag/).  INTEGRATION.md shows the ctypes binding a maintainer
 * would add on the reference side.
 *
 * Conventions: every function returns 0 on success, non-zero on failure
 * (hrag_last_error() gives the message).  Host buffers are caller-owned and C-contiguous;
 * device memory is handle-owned.  One handle drives ONE GPU (one process per GPU); a handle
 * is not thread-safe, distinct handles are independent.  There is no CPU fallback: with no
 * CUDA device hrag_create() fails.
 */
#ifndef HRAG_B200_H
#define HRAG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hrag_handle hrag_t;

/* PPR solver variants (both sweep the same CSR SpMM kernel). */
#define HRAG_PPR_POWER     0  /* z <- a P z + v            (Neumann / power iteration)        */
#define HRAG_PPR_CHEBYSHEV 1  /* Chebyshev semi-iteration on the same fixed point (default)   */

/* PPR state precision. */
#define HRAG_PPR_FP32   0     /* fp32 state, batch width ppr_batch                                   */
#define HRAG_PPR_MIXED  1     /* fp16 state (width 32) + one fp32 iterative-refinement step: same   */
                              /* accuracy as fp32, ~half the gathered bytes per query; batches of   */
                              /* <= 16 columns, and dampings whose single refinement round cannot   */
                              /* reach `tol`, run the fp32 solver                                   */

/* Similarity precision modes. */
#define HRAG_SIM_FP32     0   /* SIMT fp32 FMA kernel (exact fp32 products)                  */
#define HRAG_SIM_BF16X3   1   /* tcgen05 bf16 hi/lo split, all 4 products, fp32-faithful (default) */
#define HRAG_SIM_BF16     2   /* tcgen05 single bf16 pass (fast mode, NOT the parity mode)    */

typedef struct hrag_stats {
    double ms_sim_fact;      /* stage A: query x fact similarity (K2)                 */
    double ms_select_fact;   /* stage A: min/max + top-k facts                         */
    double ms_sim_passage;   /* stage B: query x passage similarity (K2)               */
    double ms_seed;          /* stage B: seed / reset-vector build (K3)                */
    double ms_ppr;           /* stage B: all PPR sweeps (K1)                           */
    double ms_topk;          /* stage B: passage gather + top-k (K4)                   */
    double ms_comm;          /* sharded mode: exchange time                            */
    int64_t ppr_sweeps;      /* sweeps executed since the last reset                   */
    int64_t ppr_columns;     /* sum over sweeps of the batch width B                   */
    int64_t kernel_launches; /* kernels of this library launched since the last reset  */
    int64_t h2d_bytes;
    int64_t d2h_bytes;
    double ppr_residual;     /* mixed solver, last call: measured relative L1 residual of the fp16 first solve */
    double ppr_error_bound;  /* ... times the predicted contraction of the refinement round (a-posteriori    */
                             /* bound on the relative L1 error of the PPR vectors of that call)              */
} hrag_stats_t;

const char* hrag_last_error(void);
const char* hrag_version(void);

/* Binds a handle to device_ids[0].  n_devices must be 1: multi-GPU runs use one process
 * (and one handle) per GPU, joined by hrag_comm_init().  shard_mode: 0 = replicas
 * (every rank holds the whole graph), 1 = node-range sharding. */
int hrag_create(const int* device_ids, int n_devices, int shard_mode, hrag_t** out);
void hrag_destroy(hrag_t* h);

/* Node-range sharding (SURVEY.md 8(e)): fills a 128-byte NCCL unique id (rank 0), then
 * every rank joins.  The id travels through the host's own process group. */
int hrag_comm_unique_id(void* id128);
int hrag_comm_init(hrag_t* h, const void* id128, int rank, int world);

/* Optional, before the graph load: rank r owns rows [bounds[r], bounds[r + 1]) (bounds[0] = 0, bounds[world] = N) instead
 * of equal row counts -- a partition balanced by work (non-zeros + 4 per row) keeps the ranks in step when some row
 * ranges are much denser than others (the passage rows).  hrag_load_graph_coo derives it by itself (every rank sees the
 * whole edge list); a caller of hrag_load_graph_csr passes it explicitly. */
int hrag_comm_set_row_bounds(hrag_t* h, const int64_t* bounds, int world);

/* Fused sweep + exchange for node-range sharding (after hrag_comm_init and the graph load): every
 * rank exports one 64-byte CUDA IPC handle of its PPR state, the host gathers the `world` handles
 * (rank order) and every rank imports them.  From then on the mixed-precision sweep stores its output
 * rows straight into the peers' buffers over NVLink and publishes an epoch flag -- no all-gather. */
int hrag_p2p_export(hrag_t* h, void* handle64);
int hrag_p2p_import(hrag_t* h, const void* handles, int world);

/* The graph HippoRAG.run_ppr walks (HippoRAG.py:1709-1749) as the CSR of P = W D^-1:
 * row i lists (j, W[i,j]/s_j) of the summed symmetric weights of the igraph multigraph that
 * add_new_edges builds (HippoRAG.py:1189-1223).  With node-range sharding a rank passes the
 * rows [row_lo, row_hi) it owns (row_ptr has row_hi-row_lo+1 entries, columns stay global);
 * replicas pass row_lo = 0, row_hi = n_nodes. */
int hrag_load_graph_csr(hrag_t* h, int64_t n_nodes, int64_t row_lo, int64_t row_hi, int64_t nnz,
                        const int64_t* row_ptr, const int32_t* col, const float* val);

/* Same graph from the igraph-style undirected multigraph edge list itself
 * (graph.get_edgelist() + graph.es["weight"]): every edge (src, dst, w) contributes w to W[src,dst]
 * and W[dst,src]; parallel edges sum (add_fact_edges emits (s,o) and (o,s), HippoRAG.py:907-910);
 * edges with w <= 0 carry nothing; columns are divided by the vertex strength.  The library builds
 * the CSR on the host (no scipy needed by a C caller).  With node-range sharding every rank passes
 * the full edge list and keeps its own row range. */
int hrag_load_graph_coo(hrag_t* h, int64_t n_nodes, int64_t n_edges, const int32_t* src, const int32_t* dst,
                        const double* w);

/* Integer tables equivalent to the dicts prepare_retrieval_objects builds
 * (HippoRAG.py:1287-1389): passage_vid[p] = passage_node_idxs[p] (:1333);
 * fact_subj_vid / fact_obj_vid = node_name_to_vertex_idx["entity-"+md5(phrase)] of each
 * fact's subject / object, -1 when absent (:1591-1597); ent_chunk_count[v] =
 * len(ent_node_to_chunk_ids[key]) (:1598-1601, 0 when absent). */
int hrag_load_tables(hrag_t* h, int64_t n_passages, const int32_t* passage_vid, int64_t n_facts,
                     const int32_t* fact_subj_vid, const int32_t* fact_obj_vid,
                     const int32_t* ent_chunk_count);

/* fact_embeddings (which = 0, HippoRAG.py:1345) / passage_embeddings (which = 1, :1343):
 * [rows, dim] fp32, C order.  on_device != 0: emb is a device pointer. */
int hrag_load_embeddings(hrag_t* h, int which, int64_t rows, int32_t dim, const float* emb,
                         int on_device);

/* Streamed upload for a matrix too large to keep in fp32 next to its bf16 hi/lo planes (BASELINE config #5:
 * 27.5 M facts x 1024 = 113 GB of fp32): _begin allocates only the planes of the tensor-core similarity
 * (rows x dim x 4 bytes); every _chunk converts fp32 rows [row0, row0 + n_rows) (host or device pointer) and
 * forgets them.  HRAG_SIM_FP32 is then unavailable for that matrix.  With node-range sharding a rank keeps
 * only the rows of its own fact slice and ignores the rest of a chunk. */
int hrag_load_embeddings_begin(hrag_t* h, int which, int64_t rows, int32_t dim);
int hrag_load_embeddings_chunk(hrag_t* h, int which, int64_t row0, int64_t n_rows, const float* emb,
                               int on_device);

/* Engine knobs that are not BaseConfig fields (SURVEY.md 5).  ppr_iters > 0 pins the sweep count of the
 * fp32 solver; by default it is derived from the damping factor (see hrag_stage_b). */
int hrag_set_options(hrag_t* h, int ppr_method, int ppr_iters, int ppr_batch, int sim_mode);
/* precision: HRAG_PPR_FP32 / HRAG_PPR_MIXED (-1 keeps); sweeps1 / sweeps2 > 0 pin the fp16 Chebyshev sweeps
 * before / after the residual step of the mixed solver (default: derived from damping, 8 / 7 at 0.5). */
int hrag_set_ppr_precision(hrag_t* h, int precision, int sweeps1, int sweeps2);

/* Stage A = get_fact_scores + the argsort of rerank_facts (HippoRAG.py:1427-1465,
 * 1683-1688) for B queries: top_idx[b, :] = the k best fact rows (best first; tie -> lower
 * row), top_score = their min-max-normalised scores (misc_utils.py:130-139), n_valid[b] =
 * min(k, n_facts).  k = linking_top_k (config_utils.py:184) in [1, 32]: k <= 8 is selected in the GEMM
 * epilogue, larger k by an exact radix select on the materialised scores.  Host buffers. */
int hrag_stage_a(hrag_t* h, int32_t B, const float* q_fact, int32_t k, int32_t* top_idx,
                 float* top_score, int32_t* n_valid);

/* Stage B = dense_passage_retrieval + graph_search_with_fact_entities + run_ppr + the slice
 * in _build_retrieval_result (HippoRAG.py:1467-1502, 1544-1656, 1709-1749, 501-507) for B
 * queries.  kept_fact_idx[b, :] are the fact rows that survived the recognition-memory
 * filter (-1 padded), kept_fact_score their normalised scores; a query with no kept fact or
 * dpr_only[b] != 0 takes the DPR fallback (:467-469).  out_ids index passage_node_keys
 * order (:1745), out_scores are PPR probabilities (or min-maxed DPR scores on fallback),
 * sorted by (score desc, id asc).  k_facts <= 32.  Host buffers.
 *
 * iters, tol: PRPACK iterates to 1e-10 whatever the damping (HippoRAG.py:1736-1743; damping is
 * config_utils.py:192).  Here tol = requested relative L1 accuracy of each PPR vector (0 = 1e-6, the level
 * the fp32 outputs can show) and the sweep counts are DERIVED from it: the iteration operator has its
 * spectrum in [-damping, damping], so Chebyshev contracts by damping / (1 + sqrt(1 - damping^2)) per sweep
 * (14 fp32 sweeps, or 8 + 1 + 7 fp16 sweeps with refinement, at damping 0.5; 32 fp32 sweeps at 0.85).
 * iters > 0 pins the count instead.  The mixed solver measures the residual of its first solve and the call
 * FAILS (status 4) when residual x predicted contraction misses 10 x tol. */
int hrag_stage_b(hrag_t* h, int32_t B, const float* q_pass, const int32_t* kept_fact_idx,
                 const float* kept_fact_score, int32_t k_facts, const uint8_t* dpr_only,
                 float damping, float passage_node_weight, int32_t link_top_k, int32_t topk,
                 int32_t iters, float tol, int32_t* out_ids, float* out_scores);

/* The rule hrag_stage_b / hrag_ppr apply to (damping, tol, iters) for a batch of `batch` columns with the default engine
 * options, as a pure host function (no device needed): which solver runs (use_mixed: fp16 state + refinement, batches > 16
 * whose single refinement round reaches tol), the fp32 solver's sweep count, the mixed solver's two counts, and the
 * predicted relative L1 error of the result. */
int hrag_plan_sweeps(float damping, float tol, int32_t iters, int32_t batch, int32_t* use_mixed, int32_t* fp32_sweeps,
                     int32_t* mixed_sweeps1, int32_t* mixed_sweeps2, double* predicted_error);

/* Whole retrieve() loop body for B queries with the identity recognition-memory filter,
 * inputs and outputs resident in HBM (device pointers): the device-timed benchmark leg. */
int hrag_retrieve_resident(hrag_t* h, int32_t B, const float* d_q_fact, const float* d_q_pass,
                           float damping, float passage_node_weight, int32_t link_top_k,
                           int32_t topk, int32_t iters, float tol, int32_t* d_out_ids, float* d_out_scores);

/* run_ppr's numeric core (HippoRAG.py:1735-1743) for B reset vectors: reset is [B, N]
 * (host), NaN/negative entries count as 0; out is [B, N] probabilities.  iters / tol as in hrag_stage_b. */
int hrag_ppr(hrag_t* h, int32_t B, const float* reset, float damping, int32_t iters, float tol, float* out);

/* Full score vectors for code that calls get_fact_scores (which = 0, HippoRAG.py:1427-1465)
 * or dense_passage_retrieval (which = 1, :1467-1502) directly: out[b, :] = min-max-normalised
 * <q[b], E[:, :]>, [B, rows] on the host. */
int hrag_similarity(hrag_t* h, int which, int32_t B, const float* q, float* out);

/* Top-k raw similarities (SURVEY.md 8(f)-2: the index-time synonymy KNN, utils/embed_utils.py:6-94
 * = blocked torch.mm + torch.topk): for each of B queries the k (<= 2048) rows of the fact
 * (which = 0) / passage (which = 1) embedding matrix with the largest dot product, sorted
 * (score desc, row asc); out_ids / out_scores are [B, k] (host), -1 / 0 padded when k > rows. */
int hrag_topk_similarity(hrag_t* h, int which, int32_t B, const float* q, int32_t k, int32_t* out_ids,
                         float* out_scores);

/* The KNN as add_synonymy_edges actually consumes it (HippoRAG.py:1003-1018: walk the neighbours in score order,
 * stop at the first score < synonymy_edge_sim_threshold or after 100 accepted ones): for each of B queries the rows
 * of embedding matrix `which` with dot product >= min_score, best first (score desc, row asc), at most kmax (<= 512) of
 * them; the rest of out_ids / out_scores [B, kmax] is -1 / 0.  The threshold is applied inside the GEMM epilogue -- the
 * [B, rows] score matrix is never written.  n_found[b] = how many rows cleared the threshold; n_found[b] > 512 means
 * the list of that query overflowed and it must be re-run through hrag_topk_similarity. */
int hrag_knn_threshold(hrag_t* h, int which, int32_t B, const float* q, float min_score, int32_t kmax,
                       int32_t* out_ids, float* out_scores, int32_t* n_found);

/* K1 micro-benchmark: runs `sweeps` SpMM sweeps at batch width B on resident synthetic
 * state and returns the average milliseconds per sweep (CUDA events on the launch stream).
 * method: 0 power / 1 Chebyshev (fp32 state), 2 fp16 state with a dense rhs, 3 fp16 state with the
 * compact rhs of stage B (needs hrag_load_tables). */
int hrag_bench_sweep(hrag_t* h, int32_t B, int32_t sweeps, int32_t method, float* ms_per_sweep);

/* Profiling switches (-1 keeps): k5_debug = timing probes of the fused exchange (bit 0: no per-CTA system fence,
 * bit 1: no peer stores -- results are INVALID with either; bit 2: push the row blocks with LSU stores instead of
 * TMA bulk copies -- valid, slower). */
int hrag_set_tuning(hrag_t* h, int k5_debug);

/* The CUDA stream (cudaStream_t) every kernel and copy of this handle is issued on, so a
 * caller can bracket calls with its own CUDA events. */
void* hrag_stream(hrag_t* h);

int hrag_get_stats(hrag_t* h, hrag_stats_t* out);
int hrag_reset_stats(hrag_t* h);
/* Raw device buffers for tests/benchmarks: which = 0 fact scores of the last stage A
 * sub-batch, 1 passage scores of the last stage B sub-batch. */
int hrag_debug_copy(hrag_t* h, int which, float* host_out, int64_t max_elems, int64_t* n_written);
/* keep != 0: stage A materialises the fact score matrix even in the tensor-core modes (whose
 * default epilogue selects min/max/top-k in registers and never writes scores). */
int hrag_debug_keep_scores(hrag_t* h, int keep);

#ifdef __cplusplus
}
#endif
#endif /* HRAG_B200_H */
