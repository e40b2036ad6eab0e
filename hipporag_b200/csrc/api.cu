// C ABI of libhrag_b200.so (declared in include/hrag_b200.h): handle, uploads, and the
// stage orchestration that stands in for the body of HippoRAG.retrieve()'s per-query loop
// (reference HippoRAG.py:459-480) -- batched, on one B200, all intermediate state in HBM.
//
// HBM layout per handle (N nodes, P passages, F facts, d dims; DESIGN.md section 3):
//   graph     row_ptr int32[n_rows+1], cv int2[nnz] {col, fp32 bits of P[i,j]}, row_order int32[n_rows]   (resident)
//   tables    passage_vid[P], fact_subj/obj[F], ent_chunk_count[N], slot_map[2][N] (node -> rhs slot)       (resident)
//   emb       bf16 hi/lo planes [rows, d] x 2 (tcgen05 similarity); fp32 [rows, d] only when uploaded whole  (resident)
//   state     mixed solver: H0..H3, H0b [N, 32] fp16 in one IPC-exportable slab; fp32 solver: V, XA, XC [N, B] fp32
//   rhs       compact: Vc [P + 2048, 32] fp32 (exact v) + R16 [P + 2048, 32] fp16 (scaled), two sets (double-buffered)
//   scores    S_pass [chunk, P] fp32; fact scores are never materialised in the fused modes (72 B per query x tile)
// Streams: `stream` runs the similarity, the solves and the selection; `stream2` builds the compact right-hand side of
// sub-batch i + 1 while sub-batch i is being solved.  On one GPU a sub-batch's solve is replayed as a CUDA graph.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <vector>

#include "../../include/hrag_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace hrag {

static thread_local std::string g_error;
void set_error(const std::string& msg) { g_error = msg; }

// ---- NCCL through dlopen: only sharded runs need it ---------------------------------------
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t,
                              cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int load_nccl() {
    if (g_nccl.lib) return 0;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.lib) break;
    }
    HRAG_CHECK(g_nccl.lib != nullptr, "cannot dlopen libnccl.so.2 (needed for node-range sharding)");
#define HRAG_SYM(field, name)                                                         \
    *(void**)(&g_nccl.field) = dlsym(g_nccl.lib, name);                               \
    HRAG_CHECK(g_nccl.field != nullptr, std::string("libnccl lacks ") + name)
    HRAG_SYM(GetUniqueId, "ncclGetUniqueId");
    HRAG_SYM(CommInitRank, "ncclCommInitRank");
    HRAG_SYM(CommDestroy, "ncclCommDestroy");
    HRAG_SYM(AllGather, "ncclAllGather");
    HRAG_SYM(AllReduce, "ncclAllReduce");
    HRAG_SYM(Broadcast, "ncclBroadcast");
    HRAG_SYM(GroupStart, "ncclGroupStart");
    HRAG_SYM(GroupEnd, "ncclGroupEnd");
    HRAG_SYM(GetErrorString, "ncclGetErrorString");
#undef HRAG_SYM
    return 0;
}
#define HRAG_NCCL(expr)                                                                        \
    do {                                                                                       \
        ncclResult_t _r = (expr);                                                              \
        if (_r != ncclSuccess) {                                                               \
            ::hrag::set_error(std::string(#expr) + " -> " + g_nccl.GetErrorString(_r));        \
            return 3;                                                                          \
        }                                                                                      \
    } while (0)

static std::atomic<int64_t> g_buf_generation{0};   // bumped by every (re)allocation (any handle, any thread): captured CUDA graphs hold raw pointers
struct Buf {
    void* p = nullptr;
    size_t cap = 0;
    bool view = false;        // points into another allocation (the mixed solver's slab): never freed here
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        HRAG_CHECK(!view, "internal: a slab view cannot grow");
        g_buf_generation += 1;
        if (p) HRAG_CUDA(cudaFree(p));
        p = nullptr; cap = 0;
        HRAG_CUDA(cudaMalloc(&p, bytes));
        cap = bytes;
        return 0;
    }
    void release() { if (p && !view) cudaFree(p); p = nullptr; cap = 0; view = false; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

enum Stage { ST_SIM_FACT = 0, ST_SEL_FACT, ST_SIM_PASS, ST_SEED, ST_PPR, ST_TOPK, ST_COMM, ST_COUNT };
struct Span { int stage; cudaEvent_t a, b; };

}  // namespace hrag

using namespace hrag;

struct hrag_handle {
    int device = 0;
    int shard_mode = 0;
    int rank = 0, world = 1;
    ncclComm_t comm = nullptr;
    cudaStream_t stream = nullptr;

    PprGraph g;
    int64_t chunk_rows = 0;      // rows per rank (sharded) = ceil(N / world)
    std::vector<int64_t> row_bounds;   // optional [world + 1]: rank r owns rows [row_bounds[r], row_bounds[r + 1]) -- a
                                       // work-balanced partition (non-zeros + 4 per row) instead of equal row counts
    SeedTables t;
    float* emb[2] = {nullptr, nullptr};
    bool emb_owned[2] = {false, false};
    void* emb_hi[2] = {nullptr, nullptr};   // bf16 split of emb for the tcgen05 path
    void* emb_lo[2] = {nullptr, nullptr};
    int num_sms = 148;
    int64_t emb_rows[2] = {0, 0};   // rows held by THIS handle (node-range sharding: the rank's slice of the facts)
    int64_t fact_row_lo = 0;        // first global fact row of the local slice
    int64_t n_facts_global = 0;
    int dim = 0;

    int ppr_method = HRAG_PPR_CHEBYSHEV;
    int ppr_iters = 0;    // 0 = derived from damping / tol (plan_sweeps): 14 Chebyshev sweeps at damping 0.5
    int ppr_batch = 16;
    int sim_mode = HRAG_SIM_BF16X3;
    bool keep_fact_scores = false;   // debugging: materialise S_fact even in tensor-core modes
    int ppr_precision = HRAG_PPR_MIXED;   // applies to batches of > 16 queries; smaller ones run fp32
    int mixed_m1 = 0, mixed_m2 = 0;   // 0 = derived from damping (8 / 7 at damping 0.5)
    double check_tol = 0.0, check_kappa = 0.0;   // > 0: this call's mixed solves are verified in resolve_spans
    float last_rho = 0.f;             // measured relative L1 residual of the fp16 first solve (last call)
    float last_bound = 0.f;           // a-posteriori bound on the relative L1 error of the last mixed call

    Buf V, XA, XC, partials, sums, S_fact, S_pass, mm_fact, mm_pass, mode;
    Buf d_q, d_q2, d_top_idx, d_top_score, d_nvalid, d_kept_idx, d_kept_score, d_dpr, d_out_ids, d_out_scores;
    Buf d_reset, d_scores, q_hi, q_lo, seed_vid, seed_w, H[4], mixed_aux, part_mm, part_keys;
    Buf xr_mm, xr_keys;             // fact-sharded stage A: [world, Bq] min/max and [world, Bq, 8] best keys
    // mixed solver, double-buffered per-sub-batch inputs (set s: x0 = H[0] / H0b, scales mixed_aux / mixed_aux1,
    // compact rhs Vc[s] / R16[s] addressed through slot_map[s]): stream2 prepares sub-batch i+1 while `stream`
    // sweeps sub-batch i
    Buf H0b, mixed_aux1, prep_scratch;
    Buf slot_map[2], slot_vid[2], Vc[2], R16[2], rho;
    bool slot_maps_valid = false;
    // CUDA graphs of the mixed solve, one per (buffer set, sweep plan); `graph_generation` changes whenever anything a
    // captured launch depends on does (graph / tables reload, state reallocation, tuning switches)
    struct SolveGraph {
        const void *x0 = nullptr, *slot_map = nullptr, *rhs16 = nullptr, *vexact = nullptr;
        int m1 = 0, m2 = 0;
        float alpha = 0.f;
        int64_t generation = 0;
        cudaGraphExec_t exec = nullptr;
        void *X0 = nullptr, *D = nullptr;
        int64_t sweeps = 0, columns = 0, launches = 0;
    };
    std::vector<SolveGraph> solve_graphs;
    int64_t graph_generation = 0;
    int k5_debug = 0;                          // profiling switches of the fused exchange (SweepSync::debug)
    unsigned int* d_done_ctr = nullptr;
    // one allocation [H0 | H1 | H2 | H3 | H0b | flags] so a single IPC handle exposes every buffer a peer
    // sweep may have to write into (K5, fused exchange for node-range sharding)
    void* slab = nullptr;
    size_t slab_hb = 0;                       // bytes of one fp16 state buffer inside the slab
    bool p2p = false;
    void* peer_slab[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    unsigned long long epoch = 0;             // exchange epochs signalled so far (same sequence on every rank)
    int* d_p2p_err = nullptr;
    cudaStream_t stream2 = nullptr;
    cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_released[2] = {nullptr, nullptr}, ev_inputs = nullptr;
    int64_t last_fact_rows = 0, last_pass_rows = 0;

    hrag_stats_t stats{};
    std::vector<hrag::Span> spans;
    std::vector<cudaEvent_t> pool;
};

namespace {

cudaEvent_t get_event(hrag_t* h) {
    if (!h->pool.empty()) { cudaEvent_t e = h->pool.back(); h->pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
struct StageTimer {
    hrag_t* h; int idx;
    StageTimer(hrag_t* h_, int stage) : h(h_) {
        hrag::Span s{stage, get_event(h), get_event(h)};
        cudaEventRecord(s.a, h->stream);
        h->spans.push_back(s);
        idx = (int)h->spans.size() - 1;
    }
    ~StageTimer() { cudaEventRecord(h->spans[idx].b, h->stream); }
};
}  // namespace

namespace {

int resolve_spans(hrag_t* h) {
    HRAG_CUDA(cudaStreamSynchronize(h->stream));
    if (h->p2p && h->d_p2p_err) {
        int err = 0;
        HRAG_CUDA(cudaMemcpy(&err, h->d_p2p_err, sizeof(int), cudaMemcpyDeviceToHost));
        if (err != 0) HRAG_CUDA(cudaMemset(h->d_p2p_err, 0, sizeof(int)));   // report once; this call's results are invalid
        HRAG_CHECK(err == 0, "node-range sharding: a peer GPU never published its rows (fused exchange timed out); "
                             "the results of this call are invalid");
    }
    if (h->check_tol > 0.0 && h->rho.p) {
        // a-posteriori check of the mixed solver: rho = measured relative L1 residual of the fp16 first solve (max
        // over every column solved in this call); the refinement round contracts it by kappa (plan_sweeps)
        float rho = 0.f;
        HRAG_CUDA(cudaMemcpy(&rho, h->rho.p, sizeof(float), cudaMemcpyDeviceToHost));
        HRAG_CUDA(cudaMemset(h->rho.p, 0, sizeof(float)));
        const double tol = h->check_tol, kappa = h->check_kappa;
        h->check_tol = h->check_kappa = 0.0;
        h->last_rho = rho;
        h->last_bound = (float)(rho * kappa);
        if (!(rho * kappa <= 10.0 * tol)) {
            set_error("PPR (mixed solver): measured relative residual " + std::to_string(rho) + " x predicted contraction " +
                      std::to_string(kappa) + " misses tol " + std::to_string(tol) +
                      " -- pass more sweeps (iters) or use HRAG_PPR_FP32");
            return 4;
        }
    }
    double* slots[ST_COUNT] = {&h->stats.ms_sim_fact, &h->stats.ms_select_fact, &h->stats.ms_sim_passage,
                               &h->stats.ms_seed, &h->stats.ms_ppr, &h->stats.ms_topk, &h->stats.ms_comm};
    for (auto& s : h->spans) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, s.a, s.b);
        *slots[s.stage] += ms;
        h->pool.push_back(s.a);
        h->pool.push_back(s.b);
    }
    h->spans.clear();
    h->stats.kernel_launches = launches_since_reset();
    return 0;
}

int64_t pad4(int64_t x) { return (x + 3) & ~(int64_t)3; }

int round_batch(int b) {  // PPR batch widths the sweep kernel is instantiated for
    if (b <= 4) return 4;
    if (b <= 8) return 8;
    if (b <= 16) return 16;
    if (b <= 32) return 32;
    return 64;
}

size_t state_rows(hrag_t* h) {
    return (size_t)(h->world > 1 && h->row_bounds.empty() ? h->chunk_rows * h->world : h->g.n_global);
}
void owned_rows(const hrag_t* h, int64_t n_nodes, int64_t* lo, int64_t* hi) {
    if (h->world <= 1) { *lo = 0; *hi = n_nodes; return; }
    if (!h->row_bounds.empty()) { *lo = h->row_bounds[h->rank]; *hi = h->row_bounds[h->rank + 1]; return; }
    const int64_t chunk = ceil_div(n_nodes, h->world);
    *lo = std::min<int64_t>(n_nodes, h->rank * chunk);
    *hi = std::min<int64_t>(n_nodes, (h->rank + 1) * chunk);
}
// rank r gets rows [b[r], b[r + 1]) with equal shares of cost = non-zeros + 4 per row (the epilogue streams of a row
// cost about as much as four gathers); a contiguous split by row COUNT gives the rank that holds the passage rows
// (35 non-zeros each on the synthetic graphs, 12 elsewhere) 1.4x (2 ranks) to 2.3x (8 ranks) the work of the others
std::vector<int64_t> balanced_bounds(const int64_t* row_ptr, int64_t n_nodes, int world) {
    std::vector<int64_t> b((size_t)world + 1, n_nodes);
    b[0] = 0;
    const double total = (double)row_ptr[n_nodes] + 4.0 * (double)n_nodes;
    int64_t r = 0;
    for (int k = 1; k < world; ++k) {
        const double want = total * k / world;
        while (r < n_nodes && (double)row_ptr[r] + 4.0 * (double)r < want) ++r;
        b[(size_t)k] = r;
    }
    return b;
}

int ensure_state(hrag_t* h, int B) {
    const size_t bytes = state_rows(h) * B * sizeof(float);
    HRAG_TRY(h->V.ensure(bytes));
    HRAG_TRY(h->XA.ensure(bytes));
    HRAG_TRY(h->XC.ensure(bytes));
    HRAG_TRY(h->partials.ensure((size_t)ppr_sweep_partial_rows(h->g, B) * B * sizeof(float)));
    HRAG_TRY(h->sums.ensure(64 * sizeof(double)));
    return 0;
}

int ensure_state_mixed(hrag_t* h) {
    const size_t rows = state_rows(h);
    const size_t hb = rows * 32 * 2;
    if (h->slab == nullptr || h->slab_hb != hb) {
        HRAG_CHECK(!h->p2p, "internal: the state slab cannot change after hrag_p2p_import");
        if (h->slab) HRAG_CUDA(cudaFree(h->slab));
        h->slab = nullptr;
        HRAG_CUDA(cudaMalloc(&h->slab, 5 * hb + 256));
        HRAG_CUDA(cudaMemset(static_cast<char*>(h->slab) + 5 * hb, 0, 256));      // epoch flags
        h->slab_hb = hb;
        hrag::Buf* views[5] = {&h->H[0], &h->H[1], &h->H[2], &h->H[3], &h->H0b};
        for (int i = 0; i < 5; ++i) {
            views[i]->release();
            views[i]->p = static_cast<char*>(h->slab) + (size_t)i * hb;
            views[i]->cap = hb;
            views[i]->view = true;
        }
        if (!h->d_p2p_err) {
            HRAG_CUDA(cudaMalloc(&h->d_p2p_err, sizeof(int)));
            HRAG_CUDA(cudaMemset(h->d_p2p_err, 0, sizeof(int)));
        }
        if (!h->d_done_ctr) {
            HRAG_CUDA(cudaMalloc(&h->d_done_ctr, sizeof(unsigned int)));
            HRAG_CUDA(cudaMemset(h->d_done_ctr, 0, sizeof(unsigned int)));
        }
        h->graph_generation += 1;
    }
    HRAG_TRY(h->partials.ensure((size_t)std::max(mixed_partial_rows(h->g), 1024) * 32 * sizeof(float)));
    HRAG_TRY(h->sums.ensure(192 * sizeof(double)));      // sums of x0, of d, of |r|, and of v (two sets)
    HRAG_TRY(h->mixed_aux.ensure(32 * sizeof(float)));   // column scales, set 0
    if (h->rho.p == nullptr) {
        HRAG_TRY(h->rho.ensure(sizeof(float)));
        HRAG_CUDA(cudaMemset(h->rho.p, 0, sizeof(float)));
    }
    return 0;
}

constexpr int kSeedSlots = kSeedSlotsPerQuery;   // 2 phrases per kept fact, <= 32 kept facts

// Compact right-hand-side buffers of stage B (two sets, see the handle) + the node -> slot tables.
int ensure_compact_rhs(hrag_t* h) {
    const size_t n_slots = (size_t)h->t.n_passages + 32 * kSeedSlots;
    for (int s = 0; s < 2; ++s) {
        HRAG_TRY(h->slot_map[s].ensure((size_t)h->g.n_global * sizeof(int)));
        HRAG_TRY(h->slot_vid[s].ensure(n_slots * sizeof(int)));
        HRAG_TRY(h->Vc[s].ensure(n_slots * 32 * sizeof(float)));
        HRAG_TRY(h->R16[s].ensure(n_slots * 32 * 2));
    }
    HRAG_TRY(h->mixed_aux1.ensure(32 * sizeof(float)));
    HRAG_TRY(h->prep_scratch.ensure((size_t)std::max(compact_rhs_partial_rows(h->t.n_passages), 1024) * 32 * sizeof(float)));
    if (!h->slot_maps_valid) {
        for (int s = 0; s < 2; ++s)
            HRAG_TRY(slot_map_build(h->g.n_global, h->t.n_passages, h->t.passage_vid, h->slot_map[s].as<int>(), h->stream));
        h->slot_maps_valid = true;
    }
    return 0;
}

// After a sweep wrote the owned rows of y: make every rank hold all rows (node-range sharding).
int exchange_rows_bytes(hrag_t* h, void* y, size_t row_bytes) {
    if (h->world == 1) return 0;
    StageTimer tm(h, ST_COMM);
    if (!h->row_bounds.empty()) {            // unequal ranges: one broadcast per owner, grouped into one NCCL operation
        HRAG_NCCL(g_nccl.GroupStart());
        for (int r = 0; r < h->world; ++r) {
            char* p = static_cast<char*>(y) + (size_t)h->row_bounds[r] * row_bytes;
            const size_t cnt = (size_t)(h->row_bounds[r + 1] - h->row_bounds[r]) * row_bytes;
            if (cnt) HRAG_NCCL(g_nccl.Broadcast(p, p, cnt, ncclInt8, r, h->comm, h->stream));
        }
        HRAG_NCCL(g_nccl.GroupEnd());
        return 0;
    }
    const size_t count = (size_t)h->chunk_rows * row_bytes;
    HRAG_NCCL(g_nccl.AllGather(static_cast<char*>(y) + (size_t)h->rank * count, y, count, ncclInt8, h->comm,
                               h->stream));
    return 0;
}
int exchange_rows(hrag_t* h, float* y, int B) { return exchange_rows_bytes(h, y, (size_t)B * sizeof(float)); }

unsigned long long* local_flags(hrag_t* h) {
    return reinterpret_cast<unsigned long long*>(static_cast<char*>(h->slab) + 5 * h->slab_hb);
}
PeerOut peers_for(hrag_t* h, void* y) {
    PeerOut po;
    if (!h->p2p) return po;
    const size_t off = static_cast<char*>(y) - static_cast<char*>(h->slab);
    for (int r = 0; r < h->world; ++r)
        if (r != h->rank) po.y[po.n++] = static_cast<char*>(h->peer_slab[r]) + off;
    return po;
}
// K5 epochs.  Every exchange point of the sharded solver is one epoch: all ranks run the same sequence, a rank
// waits until every peer has published everything up to the previous point and then publishes its own.  A sweep
// carries both halves itself (first instruction of every CTA / last CTA out); the two places where a non-sweep
// kernel touches exchanged state use the stand-alone wait / signal kernels.
SweepSync sync_for_sweep(hrag_t* h) {
    SweepSync sy;
    if (!h->p2p) return sy;
    sy.flags = local_flags(h);
    sy.need = h->epoch;
    sy.world = h->world;
    sy.rank = h->rank;
    sy.error_flag = h->d_p2p_err;
    sy.done_ctr = h->d_done_ctr;
    sy.debug = h->k5_debug;
    for (int r = 0; r < h->world; ++r)
        if (r != h->rank)
            sy.remote[sy.n_remote++] = reinterpret_cast<unsigned long long*>(static_cast<char*>(h->peer_slab[r]) +
                                                                              5 * h->slab_hb) + h->rank;
    h->epoch += 1;
    sy.epoch = h->epoch;
    return sy;
}
int p2p_wait(hrag_t* h) {
    if (!h->p2p) return 0;
    SweepSync sy = sync_for_sweep(h);
    h->epoch -= 1;                       // a pure wait publishes nothing
    sy.need = h->epoch;
    StageTimer tc(h, ST_COMM);
    return epoch_wait(sy, h->stream);
}
int p2p_signal(hrag_t* h) {
    if (!h->p2p) return 0;
    const SweepSync sy = sync_for_sweep(h);
    StageTimer tc(h, ST_COMM);
    return epoch_signal(sy, h->stream);
}
// one fp16 sweep + its exchange: fused peer stores (K5) when the peers are mapped, NCCL all-gather otherwise
int mixed_sweep_x(hrag_t* h, int mode, const void* x, const int* slot_map, const void* rhs, const float* v32,
                  const float* scale, const void* prev, void* y, float alpha, float w, float t, float* part,
                  int* n_part) {
    HRAG_TRY(mixed_sweep(h->g, mode, x, slot_map, rhs, v32, scale, prev, y, alpha, w, t, part, n_part, peers_for(h, y),
                         sync_for_sweep(h), h->stream));
    if (!h->p2p) HRAG_TRY(exchange_rows_bytes(h, y, 32 * 2));
    return 0;
}

// m Chebyshev sweeps of the fp16 solver on (I - aP) x = rhs, first iterate x_first (= rhs as a dense [N, 32]
// array); rhs itself is addressed through slot_map (null = dense).  Iterates alternate between bufA and bufC;
// *result = the last one, its column sums land in sums_out[0..32).
int mixed_cheb(hrag_t* h, const int* slot_map, const void* rhs, const void* x_first, void* bufA, void* bufC, int m,
               float alpha, void** result, double* sums_out) {
    HRAG_CHECK(m >= 1, "mixed solver: sweep count must be >= 1");
    const double rho2 = (double)alpha * (double)alpha;
    double w = 1.0;
    const void* x = x_first;
    const void* prev = nullptr;
    void* y = nullptr;
    int n_part = 0;
    for (int it = 1; it <= m; ++it) {
        const bool fin = it == m;
        float* part = fin ? h->partials.as<float>() : nullptr;
        if (it == 1) {
            y = bufA;
            HRAG_TRY(mixed_sweep_x(h, 0, x, slot_map, rhs, nullptr, nullptr, nullptr, y, alpha, 1.f, 1.f, part, &n_part));
        } else {
            w = it == 2 ? 1.0 / (1.0 - rho2 / 2.0) : 1.0 / (1.0 - rho2 * w / 4.0);
            if (it == 2) { prev = x_first; y = bufC; } else { y = const_cast<void*>(prev); }
            HRAG_TRY(mixed_sweep_x(h, 0, x, slot_map, rhs, nullptr, nullptr, prev, y, alpha, (float)w, 1.f, part, &n_part));
        }
        prev = x;
        x = y;
        h->stats.ppr_sweeps += 1;
        h->stats.ppr_columns += 32;
    }
    HRAG_TRY(colsum_reduce(h->partials.as<float>(), n_part, 32, sums_out, h->stream));   // local rows only: see dev_ppr_mixed_body
    *result = y;
    return 0;
}

constexpr float kMixedT = 64.f;    // residual scale: r ~ 5e-4 x, keeps it in fp16's normal range

// ---- sweep counts from (damping, tol) --------------------------------------------------------
// P is similar to a symmetric stochastic matrix, so the spectrum of aP is real in [-a, a]: Chebyshev
// semi-iteration contracts by sigma = a / (1 + sqrt(1 - a^2)) per sweep (0.268 at a = 0.5), the plain power
// sweep by a.  fp16 storage of the iterate leaves a relative L1 error of about kHalfNoise / (1 - a) in a
// converged fp16 solve (measured 5e-4 at a = 0.5, profiles/r1_accuracy_mixed.txt); one refinement round
// multiplies the error by kappa = that + 2 sigma^m2.
constexpr double kHalfNoise = 2.5e-4;
constexpr double kDefaultTol = 1e-6;     // relative L1 accuracy of the PPR vector when the caller passes tol <= 0
struct SweepPlan {
    bool mixed = false;
    int iters = 14;          // fp32 solver
    int m1 = 8, m2 = 7;      // mixed solver
    double kappa = 0.0;      // predicted contraction of the refinement round (mixed)
    double tol = kDefaultTol;
    bool check = false;      // verify the measured residual bound at the end of the call
};
// pure function of its arguments (exported as hrag_plan_sweeps so the rule is testable without a GPU); method:
// HRAG_PPR_CHEBYSHEV / HRAG_PPR_POWER for the fp32 solver; the *_override values are the handle's pins (0 = none)
SweepPlan plan_sweeps_raw(int method, int fp32_override, int m1_override, int m2_override, float alpha, int iters_arg,
                          float tol_arg, bool want_mixed) {
    SweepPlan p;
    const double a = alpha;
    const double sigma = method == HRAG_PPR_CHEBYSHEV ? a / (1.0 + std::sqrt(1.0 - a * a)) : a;
    p.tol = tol_arg > 0.f ? (double)tol_arg : kDefaultTol;
    // fp32 solver: truncation two decades under the target (1e-8 by default: the fp32 floor is ~1e-7)
    const double trunc = std::max(p.tol * 1e-2, 1e-10);
    p.iters = (int)std::ceil(std::log(trunc) / std::log(sigma) - 1e-9);
    if (fp32_override > 0) p.iters = fp32_override;
    if (iters_arg > 0) p.iters = iters_arg;
    p.iters = std::max(p.iters, 1);
    // mixed solver
    const double noise = kHalfNoise / (1.0 - a);
    const double sig_c = a / (1.0 + std::sqrt(1.0 - a * a));            // the fp16 solves are always Chebyshev
    p.m1 = (int)std::ceil(std::log(0.055 * noise) / std::log(sig_c) - 1e-9);
    p.m2 = (int)std::ceil(std::log(0.2 * noise) / std::log(sig_c) - 1e-9);
    if (m1_override > 0) p.m1 = m1_override;
    if (m2_override > 0) p.m2 = m2_override;
    if (iters_arg > 0) { p.m1 = iters_arg; p.m2 = std::max(1, iters_arg - 1); }
    p.m1 = std::max(p.m1, 1);
    p.m2 = std::max(p.m2, 1);
    p.kappa = noise + 2.0 * std::pow(sig_c, p.m2);
    const double e1 = noise + 2.0 * std::pow(sig_c, p.m1);
    const bool overridden = iters_arg > 0 || m1_override > 0 || m2_override > 0;
    // one refinement round must reach the target, otherwise the fp32 solver (which converges to its floor) runs
    p.mixed = want_mixed && (overridden || e1 * p.kappa <= p.tol);
    p.check = p.mixed && (!overridden || tol_arg > 0.f);
    return p;
}
SweepPlan plan_sweeps(const hrag_t* h, float alpha, int iters_arg, float tol_arg, bool want_mixed) {
    return plan_sweeps_raw(h->ppr_method, h->ppr_iters, h->mixed_m1, h->mixed_m2, alpha, iters_arg, tol_arg, want_mixed);
}

// sums layout (doubles): [0, 32) column sums of x0, [32, 64) of d, [64, 96) of |r|, [96, 160) of v (two buffer sets)
constexpr int kSumX0 = 0, kSumD = 32, kSumR = 64, kSumV = 96;

int dev_ppr_mixed_body(hrag_t* h, const SweepPlan& plan, float alpha, const int* slot_map, const float* Vexact,
                       const void* rhs16, void* x0_dense, const float* scale, const double* vsum, void** X0, void** D) {
    double* sums = h->sums.as<double>();
    HRAG_TRY(mixed_cheb(h, slot_map, rhs16, x0_dense, h->H[1].p, h->H[2].p, plan.m1, alpha, X0, sums + kSumX0));
    void* other = (*X0 == h->H[1].p) ? h->H[2].p : h->H[1].p;
    int n_part = 0;
    HRAG_TRY(mixed_sweep_x(h, 1, *X0, slot_map, nullptr, Vexact, scale, nullptr, h->H[3].p, alpha, 1.f, kMixedT,
                           h->partials.as<float>(), &n_part));
    h->stats.ppr_sweeps += 1;
    h->stats.ppr_columns += 32;
    HRAG_TRY(colsum_reduce(h->partials.as<float>(), n_part, 32, sums + kSumR, h->stream));
    HRAG_TRY(mixed_cheb(h, nullptr, h->H[3].p, h->H[3].p, x0_dense, other, plan.m2, alpha, D, sums + kSumD));
    if (h->world > 1) {      // node-range sharding: every rank summed its own rows -- ONE all-reduce for the three sums
        StageTimer tc(h, ST_COMM);
        HRAG_NCCL(g_nccl.AllReduce(sums, sums, 96, ncclDouble, ncclSum, h->comm, h->stream));
    }
    HRAG_TRY(residual_check(sums + kSumR, vsum, scale, 1.f / kMixedT, h->rho.as<float>(), h->stream));
    return 0;
}

// The solve of one sub-batch is ~20 launches whose arguments depend only on the buffer set and the sweep plan, so on a
// single GPU it is captured once per (set, plan) into a CUDA graph and replayed (one launch per sub-batch instead of ~20:
// what bounds small real graphs like MuSiQue-1k, where a sweep is a few microseconds of work).  Multi-GPU runs (epoch
// values change per sweep) take the plain path.
int dev_ppr_mixed(hrag_t* h, const SweepPlan& plan, float alpha, const int* slot_map, const float* Vexact,
                  const void* rhs16, void* x0_dense, const float* scale, const double* vsum, void** X0, void** D) {
    StageTimer tm(h, ST_PPR);
    if (h->world > 1) {
        HRAG_TRY(dev_ppr_mixed_body(h, plan, alpha, slot_map, Vexact, rhs16, x0_dense, scale, vsum, X0, D));
        return p2p_wait(h);     // the consumers of X0 / D (gather kernels) need every peer's last rows
    }
    hrag_handle::SolveGraph* sg = nullptr;
    for (auto& c : h->solve_graphs)
        if (c.x0 == x0_dense && c.slot_map == slot_map && c.rhs16 == rhs16 && c.vexact == Vexact && c.m1 == plan.m1 &&
            c.m2 == plan.m2 && c.alpha == alpha && c.generation == h->graph_generation + g_buf_generation) sg = &c;
    if (sg == nullptr) {
        if (h->solve_graphs.size() >= 8) {                       // bounded cache: drop everything stale
            HRAG_CUDA(cudaStreamSynchronize(h->stream));         // none of them may still be executing
            for (auto& c : h->solve_graphs) cudaGraphExecDestroy(c.exec);
            h->solve_graphs.clear();
        }
        hrag_handle::SolveGraph c;
        c.x0 = x0_dense; c.slot_map = slot_map; c.rhs16 = rhs16; c.vexact = Vexact; c.m1 = plan.m1; c.m2 = plan.m2;
        c.alpha = alpha; c.generation = h->graph_generation + g_buf_generation;
        const int64_t sw0 = h->stats.ppr_sweeps, col0 = h->stats.ppr_columns, l0 = launches_since_reset();
        HRAG_CUDA(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        const int rc = dev_ppr_mixed_body(h, plan, alpha, slot_map, Vexact, rhs16, x0_dense, scale, vsum, &c.X0, &c.D);
        cudaGraph_t graph = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
        HRAG_TRY(rc);
        HRAG_CUDA(ce);
        HRAG_CUDA(cudaGraphInstantiate(&c.exec, graph, 0));
        cudaGraphDestroy(graph);
        c.sweeps = h->stats.ppr_sweeps - sw0; c.columns = h->stats.ppr_columns - col0; c.launches = launches_since_reset() - l0;
        h->stats.ppr_sweeps = sw0; h->stats.ppr_columns = col0;   // nothing ran yet: counted at launch below
        count_launch((int)-c.launches);
        h->solve_graphs.push_back(c);
        sg = &h->solve_graphs.back();
    }
    HRAG_CUDA(cudaGraphLaunch(sg->exec, h->stream));
    h->stats.ppr_sweeps += sg->sweeps;
    h->stats.ppr_columns += sg->columns;
    count_launch((int)sg->launches);
    *X0 = sg->X0;
    *D = sg->D;
    return 0;
}

// Solves the PPR fixed point for the B columns of V; *result points at the final iterate
// (one of XA / XC), sums[b] = its column sums.
int dev_ppr(hrag_t* h, int B, int iters, float alpha, float** result) {
    HRAG_CHECK(iters >= 1, "ppr_iters must be >= 1");
    StageTimer tm(h, ST_PPR);
    float* V = h->V.as<float>();
    float* A = h->XA.as<float>();
    float* C = h->XC.as<float>();
    int n_part = 0;
    const float* x = V;
    const float* prev = nullptr;
    float* y = nullptr;
    double w = 1.0;
    const double rho2 = (double)alpha * (double)alpha;   // spectrum of alpha*P lies in [-alpha, alpha]
    for (int it = 1; it <= iters; ++it) {
        const bool fin = it == iters;
        if (h->ppr_method == HRAG_PPR_CHEBYSHEV && it >= 2) {
            w = it == 2 ? 1.0 / (1.0 - rho2 / 2.0) : 1.0 / (1.0 - rho2 * w / 4.0);
            if (it == 2) { prev = V; y = C; }                    // x = A
            else { y = const_cast<float*>(prev); }               // in place over x_{k-1}
            HRAG_TRY(ppr_sweep(h->g, B, x, V, prev, y, alpha, (float)w, fin ? h->partials.as<float>() : nullptr,
                               &n_part, h->stream));
            prev = x;
        } else {
            y = (it & 1) ? A : C;
            HRAG_TRY(ppr_sweep(h->g, B, x, V, nullptr, y, alpha, 1.f, fin ? h->partials.as<float>() : nullptr,
                               &n_part, h->stream));
            prev = x;
        }
        HRAG_TRY(exchange_rows(h, y, B));
        x = y;
        h->stats.ppr_sweeps += 1;
        h->stats.ppr_columns += B;
    }
    HRAG_TRY(colsum_reduce(h->partials.as<float>(), n_part, B, h->sums.as<double>(), h->stream));
    if (h->world > 1) {
        StageTimer tc(h, ST_COMM);
        HRAG_NCCL(g_nccl.AllReduce(h->sums.p, h->sums.p, B, ncclDouble, ncclSum, h->comm, h->stream));
    }
    *result = y;
    return 0;
}

int sim_dispatch(hrag_t* h, const float* dQ, int Bq, int which, float* S, int64_t ldS) {
    if (h->sim_mode == HRAG_SIM_FP32 || h->emb_hi[which] == nullptr) {   // dim % 8 != 0 has no TMA layout
        HRAG_CHECK(h->emb[which] != nullptr, "similarity: the fp32 embedding matrix was not kept (streamed upload); "
                                             "only the tensor-core modes are available");
        return sim_fp32(dQ, Bq, h->emb[which], h->emb_rows[which], h->dim, S, ldS, h->stream);
    }
    const size_t n = (size_t)Bq * h->dim;
    HRAG_TRY(h->q_hi.ensure(n * 2));
    HRAG_TRY(h->q_lo.ensure(n * 2));
    HRAG_TRY(split_bf16(dQ, (int64_t)n, h->q_hi.p, h->q_lo.p, h->stream));
    return sim_tc(h->q_hi.p, h->q_lo.p, Bq, h->emb_hi[which], h->emb_lo[which], h->emb_rows[which], h->dim,
                  h->sim_mode == HRAG_SIM_BF16X3 ? 4 : 1, S, ldS, nullptr, nullptr, h->num_sms, h->stream);
}

constexpr int kFusedTopK = 8;     // candidates the GEMM epilogue / row_minmax_topk keep in registers
bool fused_stage_a(hrag_t* h, int k) {   // tensor-core modes select facts in the GEMM epilogue (no score matrix)
    return h->sim_mode != HRAG_SIM_FP32 && h->emb_hi[0] != nullptr && !h->keep_fact_scores && k <= kFusedTopK;
}

int64_t chunk_a(hrag_t* h, int k) {
    const int64_t F = std::max<int64_t>(h->emb_rows[0], 1);
    if (fused_stage_a(h, k)) return 1024;     // partials are 72 B per (query, 256 facts): 0.8 GB at F = 2.75 M
    int64_t c = (int64_t)(4e9 / (4.0 * (double)pad4(F)));
    return std::max<int64_t>(1, std::min<int64_t>(c, 1024));
}
int64_t chunk_b(hrag_t* h) {
    const int64_t P = std::max<int64_t>(h->t.n_passages, 1);
    int64_t c = (int64_t)(4e9 / (4.0 * (double)pad4(P)));
    return std::max<int64_t>(1, std::min<int64_t>(c, 1024));
}

// Stage A on device pointers, Bq <= chunk_a.
int dev_stage_a(hrag_t* h, int Bq, const float* d_qf, int k, int* d_top_idx, float* d_top_score, int* d_nvalid) {
    const int64_t F = h->emb_rows[0];
    if ((h->world > 1 ? h->n_facts_global : F) == 0) {   // no facts: get_fact_scores returns an empty array (HippoRAG.py:1454-1456)
        HRAG_CUDA(cudaMemsetAsync(d_top_idx, 0xff, (size_t)Bq * k * sizeof(int), h->stream));
        HRAG_CUDA(cudaMemsetAsync(d_top_score, 0, (size_t)Bq * k * sizeof(float), h->stream));
        HRAG_CUDA(cudaMemsetAsync(d_nvalid, 0, (size_t)Bq * sizeof(int), h->stream));
        return 0;
    }
    const int64_t ld = pad4(F);
    HRAG_TRY(h->mm_fact.ensure((size_t)Bq * sizeof(float2)));
    if (fused_stage_a(h, k)) {
        const int nt = sim_tc_n_tiles(F);
        HRAG_TRY(h->part_mm.ensure((size_t)Bq * nt * sizeof(float2)));
        HRAG_TRY(h->part_keys.ensure((size_t)Bq * nt * 8 * sizeof(uint64_t)));
        const size_t n = (size_t)Bq * h->dim;
        HRAG_TRY(h->q_hi.ensure(n * 2));
        HRAG_TRY(h->q_lo.ensure(n * 2));
        {
            StageTimer tm(h, ST_SIM_FACT);
            HRAG_TRY(split_bf16(d_qf, (int64_t)n, h->q_hi.p, h->q_lo.p, h->stream));
            HRAG_TRY(sim_tc(h->q_hi.p, h->q_lo.p, Bq, h->emb_hi[0], h->emb_lo[0], F, h->dim,
                            h->sim_mode == HRAG_SIM_BF16X3 ? 4 : 1, nullptr, 0, h->part_mm.as<float2>(),
                            h->part_keys.as<uint64_t>(), h->num_sms, h->stream));
        }
        if (h->world > 1) {
            // facts are sharded by row range (SURVEY.md 8(e)): local GEMM + local top-8 -> all-gather of 8 candidates
            // and (min, max) per query -> the same merge kernel over the `world` candidate lists
            HRAG_TRY(h->xr_mm.ensure((size_t)h->world * Bq * sizeof(float2)));
            HRAG_TRY(h->xr_keys.ensure((size_t)h->world * Bq * 8 * sizeof(uint64_t)));
            float2* mm_all = h->xr_mm.as<float2>();
            uint64_t* keys_all = h->xr_keys.as<uint64_t>();
            {
                StageTimer tm(h, ST_SEL_FACT);
                HRAG_TRY(merge_minmax_topk_ex(h->part_mm.as<float2>(), h->part_keys.as<uint64_t>(), Bq, nt, nt, 1,
                                              h->fact_row_lo, F, 8, mm_all + (size_t)h->rank * Bq, nullptr, nullptr,
                                              nullptr, keys_all + (size_t)h->rank * Bq * 8, h->stream));
            }
            {
                StageTimer tc(h, ST_COMM);
                HRAG_NCCL(g_nccl.AllGather(mm_all + (size_t)h->rank * Bq, mm_all, (size_t)Bq * sizeof(float2), ncclInt8,
                                           h->comm, h->stream));
                HRAG_NCCL(g_nccl.AllGather(keys_all + (size_t)h->rank * Bq * 8, keys_all, (size_t)Bq * 8 * sizeof(uint64_t),
                                           ncclInt8, h->comm, h->stream));
            }
            StageTimer tm(h, ST_SEL_FACT);
            HRAG_TRY(merge_minmax_topk_ex(mm_all, keys_all, Bq, h->world, 1, Bq, 0, h->n_facts_global, k,
                                          h->mm_fact.as<float2>(), d_top_idx, d_top_score, d_nvalid, nullptr, h->stream));
            h->last_fact_rows = 0;
            return 0;
        }
        {
            StageTimer tm(h, ST_SEL_FACT);
            HRAG_TRY(merge_minmax_topk(h->part_mm.as<float2>(), h->part_keys.as<uint64_t>(), Bq, nt, F, k,
                                       h->mm_fact.as<float2>(), d_top_idx, d_top_score, d_nvalid, h->stream));
        }
        h->last_fact_rows = 0;
        return 0;
    }
    HRAG_CHECK(h->world == 1, "node-range sharding: stage A needs the tensor-core similarity with linking_top_k <= 8 "
                              "(the fact rows are sharded; the fp32 / materialised paths are single-GPU)");
    HRAG_TRY(h->S_fact.ensure((size_t)Bq * ld * sizeof(float)));
    {
        StageTimer tm(h, ST_SIM_FACT);
        HRAG_TRY(sim_dispatch(h, d_qf, Bq, 0, h->S_fact.as<float>(), ld));
    }
    {
        StageTimer tm(h, ST_SEL_FACT);
        if (k <= kFusedTopK) {
            HRAG_TRY(row_minmax_topk(h->S_fact.as<float>(), Bq, F, ld, k, h->mm_fact.as<float2>(), d_top_idx,
                                     d_top_score, d_nvalid, h->stream));
        } else {   // linking_top_k > 8 (config_utils.py:184): exact radix select on the materialised scores
            HRAG_TRY(row_minmax_topk(h->S_fact.as<float>(), Bq, F, ld, 0, h->mm_fact.as<float2>(), nullptr, nullptr,
                                     nullptr, h->stream));
            HRAG_TRY(row_topk(h->S_fact.as<float>(), Bq, F, ld, k, d_top_idx, d_top_score, h->stream));
            HRAG_TRY(topk_normalize(Bq, k, F, h->mm_fact.as<float2>(), d_top_idx, d_top_score, d_nvalid, h->stream));
        }
    }
    h->last_fact_rows = Bq;
    return 0;
}

// Stage B on device pointers, Bq <= chunk_b.
int dev_stage_b(hrag_t* h, int Bq, const float* d_qp, const int* d_kept_idx, const float* d_kept_score,
                int k_facts, const uint8_t* d_dpr, float damping, float pnw, int link_top_k, int topk,
                int iters_arg, float tol_arg, int* d_out_ids, float* d_out_scores) {
    const int P = h->t.n_passages;
    HRAG_CHECK(P > 0, "stage B: no passages loaded");
    const int64_t ld = pad4(P);
    HRAG_TRY(h->S_pass.ensure((size_t)Bq * ld * sizeof(float)));
    HRAG_TRY(h->mm_pass.ensure((size_t)Bq * sizeof(float2)));
    HRAG_TRY(h->mode.ensure((size_t)Bq * sizeof(int)));
    float* S = h->S_pass.as<float>();
    {
        StageTimer tm(h, ST_SIM_PASS);
        HRAG_TRY(sim_dispatch(h, d_qp, Bq, 1, S, ld));
        HRAG_TRY(row_minmax_topk(S, Bq, P, ld, 0, h->mm_pass.as<float2>(), nullptr, nullptr, nullptr, h->stream));
    }
    const SweepPlan plan = plan_sweeps(h, damping, iters_arg, tol_arg, h->ppr_precision == HRAG_PPR_MIXED && Bq > 16);
    const bool mixed = plan.mixed;
    const int Bp = mixed ? 32 : round_batch(std::min(h->ppr_batch, Bq));
    if (mixed) { HRAG_TRY(ensure_state_mixed(h)); HRAG_TRY(ensure_compact_rhs(h)); }
    else HRAG_TRY(ensure_state(h, Bp));
    HRAG_TRY(h->seed_vid.ensure((size_t)Bq * kSeedSlots * sizeof(int)));     // [Bq, kSeedSlots] seed slots
    HRAG_TRY(h->seed_w.ensure((size_t)Bq * kSeedSlots * sizeof(float)));
    {
        StageTimer tm(h, ST_SEED);
        HRAG_TRY(seed_entities(h->t, Bq, d_kept_idx, d_kept_score, k_facts, d_dpr, link_top_k, h->seed_vid.as<int>(),
                               h->seed_w.as<float>(), h->mode.as<int>(), h->stream));
    }
    if (k_facts == 0) {   // retrieve_dpr (HippoRAG.py:665-732): every query is a DPR query, no PPR at all
        StageTimer tm(h, ST_TOPK);
        HRAG_TRY(minmax_apply(S, Bq, P, ld, h->mm_pass.as<float2>(), h->stream));
    }
    if (mixed && k_facts > 0) {
        // Two streams: stream2 builds sub-batch i+1's compact right-hand side (passage weights + phrase seeds on
        // P + 2048 slots, its column scales, the fp16 copy and the dense first iterate) while `stream` runs the
        // sweeps of sub-batch i.
        if (plan.check) h->check_tol = std::max(h->check_tol, plan.tol), h->check_kappa = plan.kappa;
        HRAG_CUDA(cudaEventRecord(h->ev_inputs, h->stream));            // S, min/max, seed lists are ready
        HRAG_CUDA(cudaStreamWaitEvent(h->stream2, h->ev_inputs, 0));
        int it = 0;
        for (int q0 = 0; q0 < Bq; q0 += 32, ++it) {
            const int nb = std::min(32, Bq - q0);
            const int set = it & 1;
            void* x0 = set ? h->H0b.p : h->H[0].p;
            float* scale = set ? h->mixed_aux1.as<float>() : h->mixed_aux.as<float>();
            double* vsum = h->sums.as<double>() + kSumV + 32 * set;
            int* slot_map = h->slot_map[set].as<int>();
            if (it >= 2) HRAG_CUDA(cudaStreamWaitEvent(h->stream2, h->ev_released[set], 0));   // set is free again
            HRAG_TRY(compact_prepare_rhs(h->t, nb, q0, S, ld, h->mm_pass.as<float2>(), pnw, kSeedSlots,
                                         h->seed_vid.as<int>(), h->seed_w.as<float>(), damping, slot_map,
                                         h->slot_vid[set].as<int>(), h->Vc[set].as<float>(), h->R16[set].p, x0,
                                         (int64_t)h->g.n_global, h->prep_scratch.as<float>(), vsum, scale, h->stream2));
            HRAG_CUDA(cudaEventRecord(h->ev_ready[set], h->stream2));
            HRAG_CUDA(cudaStreamWaitEvent(h->stream, h->ev_ready[set], 0));
            void *X0 = nullptr, *D = nullptr;
            HRAG_TRY(dev_ppr_mixed(h, plan, damping, slot_map, h->Vc[set].as<float>(), h->R16[set].p, x0, scale, vsum,
                                   &X0, &D));
            {
                StageTimer tm(h, ST_TOPK);
                HRAG_TRY(gather_passage_scores_mixed(h->t, nb, q0, X0, D, 1.f / kMixedT, h->sums.as<double>(),
                                                     h->sums.as<double>() + 32, h->mode.as<int>(),
                                                     h->mm_pass.as<float2>(), S, ld, h->stream));
                HRAG_TRY(compact_release_slots(P, nb, q0, kSeedSlots, h->seed_vid.as<int>(), slot_map, h->stream));
            }
            HRAG_TRY(p2p_signal(h));   // peers may overwrite this rank's state buffers from here on
            HRAG_CUDA(cudaEventRecord(h->ev_released[set], h->stream));
        }
        // (every prepare was consumed by a solve on `stream`, so stream2 is drained in stream order)
    }
    for (int q0 = 0; q0 < Bq && k_facts > 0 && !mixed; q0 += Bp) {
        const int nb = std::min(Bp, Bq - q0);
        {
            StageTimer tm(h, ST_SEED);
            HRAG_CUDA(cudaMemsetAsync(h->V.p, 0, (size_t)h->g.n_global * Bp * sizeof(float), h->stream));
            HRAG_TRY(seed_passages(h->t, Bp, nb, S, ld, q0, h->mm_pass.as<float2>(), pnw, h->V.as<float>(), h->stream));
            HRAG_TRY(seed_scatter(Bp, nb, q0, h->seed_vid.as<int>(), h->seed_w.as<float>(), h->V.as<float>(),
                                  h->stream));
        }
        float* Z = nullptr;
        HRAG_TRY(dev_ppr(h, Bp, plan.iters, damping, &Z));
        StageTimer tm(h, ST_TOPK);
        HRAG_TRY(gather_passage_scores(h->t, Bp, nb, q0, Z, h->sums.as<double>(), h->mode.as<int>(),
                                       h->mm_pass.as<float2>(), S, ld, h->stream));
    }
    {
        StageTimer tm(h, ST_TOPK);
        HRAG_TRY(row_topk(S, Bq, P, ld, topk, d_out_ids, d_out_scores, h->stream));
    }
    h->last_pass_rows = Bq;
    return 0;
}

int h2d(hrag_t* h, void* dst, const void* src, size_t bytes) {
    HRAG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->stream));
    h->stats.h2d_bytes += (int64_t)bytes;
    return 0;
}
int d2h(hrag_t* h, void* dst, const void* src, size_t bytes) {
    HRAG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += (int64_t)bytes;
    return 0;
}

}  // namespace

// =================================================================================== C ABI
extern "C" {

const char* hrag_last_error(void) { return g_error.c_str(); }
const char* hrag_version(void) { return "hrag_b200 0.1 (sm_100a)"; }

int hrag_create(const int* device_ids, int n_devices, int shard_mode, hrag_t** out) {
    HRAG_CHECK(out != nullptr, "hrag_create: out is null");
    HRAG_CHECK(n_devices == 1 && device_ids != nullptr,
               "hrag_create: one handle drives one GPU (n_devices must be 1); use one process per GPU");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_error("hrag_create: no CUDA device visible -- this library has no CPU fallback");
        return 1;
    }
    HRAG_CHECK(device_ids[0] >= 0 && device_ids[0] < count, "hrag_create: bad device id");
    HRAG_CUDA(cudaSetDevice(device_ids[0]));
    cudaDeviceProp prop;
    HRAG_CUDA(cudaGetDeviceProperties(&prop, device_ids[0]));
    HRAG_CHECK(prop.major == 10, "hrag_create: this library is built for sm_100a (B200) only");
    hrag_t* h = new hrag_handle();
    h->device = device_ids[0];
    h->shard_mode = shard_mode;
    h->num_sms = prop.multiProcessorCount;
    HRAG_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    HRAG_CUDA(cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        HRAG_CUDA(cudaEventCreateWithFlags(&h->ev_ready[i], cudaEventDisableTiming));
        HRAG_CUDA(cudaEventCreateWithFlags(&h->ev_released[i], cudaEventDisableTiming));
    }
    HRAG_CUDA(cudaEventCreateWithFlags(&h->ev_inputs, cudaEventDisableTiming));
    *out = h;
    return 0;
}

void hrag_destroy(hrag_t* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    for (hrag::Buf* b : {&h->V, &h->XA, &h->XC, &h->partials, &h->sums, &h->S_fact, &h->S_pass, &h->mm_fact,
                         &h->mm_pass, &h->mode, &h->d_q, &h->d_q2, &h->d_top_idx, &h->d_top_score, &h->d_nvalid,
                         &h->d_kept_idx, &h->d_kept_score, &h->d_dpr, &h->d_out_ids, &h->d_out_scores,
                         &h->d_reset, &h->d_scores, &h->q_hi, &h->q_lo, &h->seed_vid, &h->seed_w, &h->H[0], &h->H[1],
                         &h->H[2], &h->H[3], &h->mixed_aux, &h->part_mm, &h->part_keys, &h->H0b,
                         &h->mixed_aux1, &h->prep_scratch, &h->slot_map[0], &h->slot_map[1], &h->slot_vid[0],
                         &h->slot_vid[1], &h->Vc[0], &h->Vc[1], &h->R16[0], &h->R16[1], &h->rho, &h->xr_mm, &h->xr_keys})
        b->release();
    cudaFree(h->g.row_ptr); cudaFree(h->g.cv); cudaFree(h->g.long_rows); cudaFree(h->g.long_seg_ptr);
    cudaFree(h->g.segs); cudaFree(h->g.seg_partial); cudaFree(h->g.row_order);
    cudaFree(h->t.passage_vid); cudaFree(h->t.fact_subj_vid); cudaFree(h->t.fact_obj_vid);
    cudaFree(h->t.ent_chunk_count);
    for (int i = 0; i < 2; ++i) {
        if (h->emb_owned[i]) cudaFree(h->emb[i]);
        cudaFree(h->emb_hi[i]);
        cudaFree(h->emb_lo[i]);
    }
    for (auto& c : h->solve_graphs) cudaGraphExecDestroy(c.exec);
    for (auto e : h->pool) cudaEventDestroy(e);
    for (int r = 0; r < 8; ++r) if (h->peer_slab[r]) cudaIpcCloseMemHandle(h->peer_slab[r]);
    cudaFree(h->slab);
    cudaFree(h->d_p2p_err);
    cudaFree(h->d_done_ctr);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(h->ev_ready[i]); cudaEventDestroy(h->ev_released[i]); }
    cudaEventDestroy(h->ev_inputs);
    cudaStreamDestroy(h->stream2);
    cudaStreamDestroy(h->stream);
    delete h;
}

int hrag_comm_unique_id(void* id128) {
    HRAG_TRY(load_nccl());
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    HRAG_NCCL(g_nccl.GetUniqueId(reinterpret_cast<ncclUniqueId*>(id128)));
    return 0;
}

int hrag_comm_init(hrag_t* h, const void* id128, int rank, int world) {
    HRAG_CHECK(h && id128, "hrag_comm_init: null argument");
    HRAG_CHECK(world >= 1 && rank >= 0 && rank < world, "hrag_comm_init: bad rank/world");
    HRAG_TRY(load_nccl());
    HRAG_CUDA(cudaSetDevice(h->device));
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    HRAG_NCCL(g_nccl.CommInitRank(&h->comm, world, id, rank));
    h->rank = rank;
    h->world = world;
    return 0;
}

int hrag_comm_set_row_bounds(hrag_t* h, const int64_t* bounds, int world) {
    HRAG_CHECK(h && bounds, "hrag_comm_set_row_bounds: null argument");
    HRAG_CHECK(world == h->world && world >= 1, "hrag_comm_set_row_bounds: world must match hrag_comm_init");
    HRAG_CHECK(!h->p2p, "hrag_comm_set_row_bounds: set the partition before hrag_p2p_export / import");
    HRAG_CHECK(bounds[0] == 0, "hrag_comm_set_row_bounds: bounds[0] must be 0");
    for (int r = 0; r < world; ++r) HRAG_CHECK(bounds[r] <= bounds[r + 1], "hrag_comm_set_row_bounds: bounds must not decrease");
    h->row_bounds.assign(bounds, bounds + world + 1);
    return 0;
}

int hrag_p2p_export(hrag_t* h, void* handle64) {
    HRAG_CHECK(h && handle64, "hrag_p2p_export: null argument");
    HRAG_CHECK(h->g.n_global > 0, "hrag_p2p_export: load the graph first");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    HRAG_CUDA(cudaSetDevice(h->device));
    HRAG_TRY(ensure_state_mixed(h));
    cudaIpcMemHandle_t mh;
    HRAG_CUDA(cudaIpcGetMemHandle(&mh, h->slab));
    memcpy(handle64, &mh, 64);
    return 0;
}

int hrag_p2p_import(hrag_t* h, const void* handles, int world) {
    HRAG_CHECK(h && handles, "hrag_p2p_import: null argument");
    HRAG_CHECK(world == h->world && world >= 2 && world <= 8, "hrag_p2p_import: world must match hrag_comm_init (2..8)");
    HRAG_CHECK(h->slab != nullptr, "hrag_p2p_import: call hrag_p2p_export first");
    HRAG_CUDA(cudaSetDevice(h->device));
    for (int r = 0; r < world; ++r) {
        if (r == h->rank) continue;
        cudaIpcMemHandle_t mh;
        memcpy(&mh, static_cast<const char*>(handles) + (size_t)r * 64, 64);
        HRAG_CUDA(cudaIpcOpenMemHandle(&h->peer_slab[r], mh, cudaIpcMemLazyEnablePeerAccess));
    }
    h->p2p = true;
    h->epoch = 0;
    return 0;
}

int hrag_load_graph_csr(hrag_t* h, int64_t n_nodes, int64_t row_lo, int64_t row_hi, int64_t nnz,
                        const int64_t* row_ptr, const int32_t* col, const float* val) {
    HRAG_CHECK(h && row_ptr && (nnz == 0 || (col && val)), "hrag_load_graph_csr: null argument");
    HRAG_CHECK(n_nodes > 0 && n_nodes < (int64_t)1 << 30, "hrag_load_graph_csr: n_nodes out of range");
    HRAG_CHECK(nnz >= 0 && nnz < ((int64_t)1 << 31) - 8, "hrag_load_graph_csr: nnz must fit int32");
    HRAG_CHECK(0 <= row_lo && row_lo <= row_hi && row_hi <= n_nodes, "hrag_load_graph_csr: bad row range");
    HRAG_CUDA(cudaSetDevice(h->device));
    const int n_rows = (int)(row_hi - row_lo);
    HRAG_CHECK(row_ptr[0] == 0 && row_ptr[n_rows] == nnz, "hrag_load_graph_csr: row_ptr does not span nnz");
    PprGraph& g = h->g;
    cudaFree(g.row_ptr); cudaFree(g.cv); cudaFree(g.long_rows); cudaFree(g.long_seg_ptr); cudaFree(g.segs);
    cudaFree(g.seg_partial);
    cudaFree(g.row_order);
    g = PprGraph();
    g.num_sms = h->num_sms;
    g.n_global = (int)n_nodes;
    g.row_lo = (int)row_lo;
    g.n_rows = n_rows;
    g.nnz = nnz;
    g.long_thresh = 256;
    g.max_batch = 64;
    h->chunk_rows = h->world > 1 ? ceil_div(n_nodes, h->world) : n_nodes;
    if (h->world > 1) {
        HRAG_CHECK(h->row_bounds.empty() || h->row_bounds.back() == n_nodes,
                   "hrag_load_graph_csr: hrag_comm_set_row_bounds was given bounds for a different vertex count");
        int64_t lo = 0, hi = 0;
        owned_rows(h, n_nodes, &lo, &hi);
        HRAG_CHECK(row_lo == lo && row_hi == hi,
                   "hrag_load_graph_csr: sharded ranks own rows [rank*ceil(N/world), (rank+1)*ceil(N/world)), or the range "
                   "given by hrag_comm_set_row_bounds");
    }
    std::vector<int> rp(n_rows + 1);
    std::vector<int2> cv((size_t)nnz);
    std::vector<int> long_rows, long_seg_ptr;
    std::vector<int4> segs;
    const int seg_len = 256;
    for (int r = 0; r < n_rows; ++r) {
        const int64_t s = row_ptr[r], e = row_ptr[r + 1];
        HRAG_CHECK(s <= e && e <= nnz, "hrag_load_graph_csr: row_ptr not monotone");
        rp[r] = (int)s;
        if (e - s > g.long_thresh) {
            long_rows.push_back(r);
            long_seg_ptr.push_back((int)segs.size());
            for (int64_t a = s; a < e; a += seg_len)
                segs.push_back(make_int4(r, (int)a, (int)std::min<int64_t>(e, a + seg_len), 0));
        }
    }
    rp[n_rows] = (int)nnz;
    long_seg_ptr.push_back((int)segs.size());
    for (int64_t i = 0; i < nnz; ++i) {
        HRAG_CHECK(col[i] >= 0 && col[i] < n_nodes, "hrag_load_graph_csr: column index out of range");
        int bits;
        memcpy(&bits, &val[i], 4);
        cv[(size_t)i] = make_int2(col[i], bits);
    }
    HRAG_CUDA(cudaMalloc(&g.row_ptr, (size_t)(n_rows + 1) * sizeof(int)));
    HRAG_CUDA(cudaMalloc(&g.cv, ((size_t)nnz + 2) * sizeof(int2)));   // +2 zeroed spares: never null, even with no edges
    HRAG_CUDA(cudaMemset(g.cv, 0, ((size_t)nnz + 2) * sizeof(int2)));
    HRAG_CUDA(cudaMemcpy(g.row_ptr, rp.data(), (size_t)(n_rows + 1) * sizeof(int), cudaMemcpyHostToDevice));
    if (nnz) HRAG_CUDA(cudaMemcpy(g.cv, cv.data(), (size_t)nnz * sizeof(int2), cudaMemcpyHostToDevice));
    {   // fp16 sweep: within each block of 64 rows (one CTA) order the rows by length so a warp's 8 rows match
        std::vector<int> order(n_rows);
        for (int r = 0; r < n_rows; ++r) order[r] = r;
        for (int b0 = 0; b0 < n_rows; b0 += 64) {
            const int b1 = std::min(n_rows, b0 + 64);
            std::stable_sort(order.begin() + b0, order.begin() + b1,
                             [&](int x, int y) { return rp[x + 1] - rp[x] > rp[y + 1] - rp[y]; });
        }
        HRAG_CUDA(cudaMalloc(&g.row_order, std::max<size_t>(1, order.size()) * sizeof(int)));
        if (n_rows) HRAG_CUDA(cudaMemcpy(g.row_order, order.data(), order.size() * sizeof(int), cudaMemcpyHostToDevice));
    }
    g.n_long = (int)long_rows.size();
    g.n_seg = (int)segs.size();
    if (g.n_long) {
        HRAG_CUDA(cudaMalloc(&g.long_rows, long_rows.size() * sizeof(int)));
        HRAG_CUDA(cudaMalloc(&g.long_seg_ptr, long_seg_ptr.size() * sizeof(int)));
        HRAG_CUDA(cudaMalloc(&g.segs, segs.size() * sizeof(int4)));
        HRAG_CUDA(cudaMalloc(&g.seg_partial, segs.size() * (size_t)g.max_batch * sizeof(float)));
        HRAG_CUDA(cudaMemcpy(g.long_rows, long_rows.data(), long_rows.size() * sizeof(int), cudaMemcpyHostToDevice));
        HRAG_CUDA(cudaMemcpy(g.long_seg_ptr, long_seg_ptr.data(), long_seg_ptr.size() * sizeof(int),
                             cudaMemcpyHostToDevice));
        HRAG_CUDA(cudaMemcpy(g.segs, segs.data(), segs.size() * sizeof(int4), cudaMemcpyHostToDevice));
    }
    h->V.release(); h->XA.release(); h->XC.release(); h->partials.release();
    h->slot_maps_valid = false;
    h->graph_generation += 1;
    return 0;
}

int hrag_load_graph_coo(hrag_t* h, int64_t n_nodes, int64_t n_edges, const int32_t* src, const int32_t* dst,
                        const double* w) {
    HRAG_CHECK(h && (n_edges == 0 || (src && dst && w)), "hrag_load_graph_coo: null argument");
    HRAG_CHECK(n_nodes > 0 && n_nodes < (int64_t)1 << 30 && n_edges >= 0 && n_edges < (int64_t)1 << 30,
               "hrag_load_graph_coo: sizes out of range");
    // symmetrise: (row, col, w) for both directions, keyed row-major
    struct Ent { uint64_t key; double w; };
    std::vector<Ent> e;
    e.reserve((size_t)n_edges * 2);
    for (int64_t i = 0; i < n_edges; ++i) {
        const int64_t a = src[i], b = dst[i];
        HRAG_CHECK(a >= 0 && a < n_nodes && b >= 0 && b < n_nodes, "hrag_load_graph_coo: edge endpoint out of range");
        if (!(w[i] > 0.0)) continue;                       // non-positive (and NaN) weights carry nothing
        e.push_back({((uint64_t)a << 32) | (uint64_t)b, w[i]});
        e.push_back({((uint64_t)b << 32) | (uint64_t)a, w[i]});
    }
    std::stable_sort(e.begin(), e.end(), [](const Ent& x, const Ent& y) { return x.key < y.key; });
    std::vector<int64_t> row_ptr((size_t)n_nodes + 1, 0);
    std::vector<int32_t> col;
    std::vector<double> wsum;
    col.reserve(e.size());
    wsum.reserve(e.size());
    for (size_t i = 0; i < e.size();) {                    // merge parallel edges in input order
        size_t j = i;
        double s = 0.0;
        while (j < e.size() && e[j].key == e[i].key) s += e[j++].w;
        col.push_back((int32_t)(e[i].key & 0xffffffffu));
        wsum.push_back(s);
        row_ptr[(size_t)(e[i].key >> 32) + 1] += 1;
        i = j;
    }
    for (int64_t r = 0; r < n_nodes; ++r) row_ptr[(size_t)r + 1] += row_ptr[(size_t)r];
    std::vector<double> strength((size_t)n_nodes, 0.0);    // W is symmetric: column sums = row sums
    for (int64_t r = 0; r < n_nodes; ++r)
        for (int64_t k = row_ptr[(size_t)r]; k < row_ptr[(size_t)r + 1]; ++k) strength[(size_t)r] += wsum[(size_t)k];
    std::vector<float> val(col.size());
    for (size_t k = 0; k < col.size(); ++k) val[k] = (float)(wsum[k] / strength[(size_t)col[k]]);
    int64_t lo = 0, hi = n_nodes;
    if (h->world > 1) {
        // every rank sees the whole edge list here, so all of them derive the same work-balanced partition
        h->row_bounds = balanced_bounds(row_ptr.data(), n_nodes, h->world);
        owned_rows(h, n_nodes, &lo, &hi);
    }
    const int64_t a = row_ptr[(size_t)lo], b = row_ptr[(size_t)hi];
    std::vector<int64_t> rp((size_t)(hi - lo) + 1);
    for (int64_t r = lo; r <= hi; ++r) rp[(size_t)(r - lo)] = row_ptr[(size_t)r] - a;
    return hrag_load_graph_csr(h, n_nodes, lo, hi, b - a, rp.data(), col.data() + a, val.data() + a);
}

static int upload_i32(int** dst, const int32_t* src, int64_t n) {
    cudaFree(*dst);
    *dst = nullptr;
    HRAG_CUDA(cudaMalloc(dst, std::max<size_t>(1, (size_t)n) * sizeof(int)));
    if (n) HRAG_CUDA(cudaMemcpy(*dst, src, (size_t)n * sizeof(int), cudaMemcpyHostToDevice));
    return 0;
}

int hrag_load_tables(hrag_t* h, int64_t n_passages, const int32_t* passage_vid, int64_t n_facts,
                     const int32_t* fact_subj_vid, const int32_t* fact_obj_vid, const int32_t* ent_chunk_count) {
    HRAG_CHECK(h, "hrag_load_tables: null handle");
    HRAG_CHECK(h->g.n_global > 0, "hrag_load_tables: load the graph first");
    HRAG_CHECK(n_passages >= 0 && n_passages < (int64_t)1 << 31 && n_facts >= 0, "hrag_load_tables: bad sizes");
    HRAG_CUDA(cudaSetDevice(h->device));
    const int N = h->g.n_global;
    for (int64_t p = 0; p < n_passages; ++p)
        HRAG_CHECK(passage_vid[p] >= 0 && passage_vid[p] < N, "hrag_load_tables: passage_vid out of range");
    for (int64_t f = 0; f < n_facts; ++f)
        HRAG_CHECK(fact_subj_vid[f] < N && fact_obj_vid[f] < N, "hrag_load_tables: fact vertex id out of range");
    h->slot_maps_valid = false;
    h->graph_generation += 1;
    h->t.n_nodes = N;
    h->t.n_passages = (int)n_passages;
    h->t.n_facts = n_facts;
    HRAG_TRY(upload_i32(&h->t.passage_vid, passage_vid, n_passages));
    HRAG_TRY(upload_i32(&h->t.fact_subj_vid, fact_subj_vid, n_facts));
    HRAG_TRY(upload_i32(&h->t.fact_obj_vid, fact_obj_vid, n_facts));
    HRAG_TRY(upload_i32(&h->t.ent_chunk_count, ent_chunk_count, N));
    return 0;
}

int hrag_load_embeddings(hrag_t* h, int which, int64_t rows, int32_t dim, const float* emb, int on_device) {
    HRAG_CHECK(h && (which == 0 || which == 1), "hrag_load_embeddings: which must be 0 (fact) or 1 (passage)");
    HRAG_CHECK(rows >= 0 && dim > 0 && dim % 4 == 0, "hrag_load_embeddings: dim must be a positive multiple of 4");
    HRAG_CHECK(rows == 0 || emb != nullptr, "hrag_load_embeddings: null embeddings");
    HRAG_CHECK(h->dim == 0 || h->dim == dim || h->emb_rows[1 - which] == 0,
               "hrag_load_embeddings: fact and passage embeddings must share dim");
    HRAG_CUDA(cudaSetDevice(h->device));
    if (h->emb_owned[which]) cudaFree(h->emb[which]);
    cudaFree(h->emb_hi[which]);
    cudaFree(h->emb_lo[which]);
    h->emb[which] = nullptr;
    h->emb_hi[which] = h->emb_lo[which] = nullptr;
    h->emb_owned[which] = false;
    h->dim = dim;
    if (which == 0) {
        h->n_facts_global = rows;
        h->fact_row_lo = 0;
        if (h->world > 1) {          // node-range sharding: this rank keeps fact rows [rank * ceil(F / world), ...)
            const int64_t chunk = ceil_div(rows, h->world);
            const int64_t lo = std::min<int64_t>(rows, h->rank * chunk), hi = std::min<int64_t>(rows, (h->rank + 1) * chunk);
            h->fact_row_lo = lo;
            emb += (size_t)lo * dim;
            rows = hi - lo;
        }
    }
    h->emb_rows[which] = rows;
    if (rows == 0) return 0;
    if (on_device) {
        h->emb[which] = const_cast<float*>(emb);   // caller keeps it alive
    } else {
        HRAG_CUDA(cudaMalloc(&h->emb[which], (size_t)rows * dim * sizeof(float)));
        h->emb_owned[which] = true;
        HRAG_CUDA(cudaMemcpy(h->emb[which], emb, (size_t)rows * dim * sizeof(float), cudaMemcpyHostToDevice));
    }
    if (dim % 8 == 0) {   // bf16 hi/lo split for the tcgen05 similarity kernel
        const size_t n = (size_t)rows * dim;
        HRAG_CUDA(cudaMalloc(&h->emb_hi[which], n * 2));
        HRAG_CUDA(cudaMalloc(&h->emb_lo[which], n * 2));
        HRAG_TRY(split_bf16(h->emb[which], (int64_t)n, h->emb_hi[which], h->emb_lo[which], h->stream));
        HRAG_CUDA(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

int hrag_load_embeddings_begin(hrag_t* h, int which, int64_t rows, int32_t dim) {
    HRAG_CHECK(h && (which == 0 || which == 1), "hrag_load_embeddings_begin: which must be 0 (fact) or 1 (passage)");
    HRAG_CHECK(rows > 0 && dim > 0 && dim % 8 == 0, "hrag_load_embeddings_begin: rows > 0 and dim a multiple of 8");
    HRAG_CHECK(h->dim == 0 || h->dim == dim || h->emb_rows[1 - which] == 0,
               "hrag_load_embeddings_begin: fact and passage embeddings must share dim");
    HRAG_CUDA(cudaSetDevice(h->device));
    if (h->emb_owned[which]) cudaFree(h->emb[which]);
    cudaFree(h->emb_hi[which]);
    cudaFree(h->emb_lo[which]);
    h->emb[which] = nullptr;
    h->emb_hi[which] = h->emb_lo[which] = nullptr;
    h->emb_owned[which] = false;
    h->dim = dim;
    int64_t lo = 0, hi = rows;
    if (which == 0) {
        h->n_facts_global = rows;
        if (h->world > 1) {
            const int64_t chunk = ceil_div(rows, h->world);
            lo = std::min<int64_t>(rows, h->rank * chunk);
            hi = std::min<int64_t>(rows, (h->rank + 1) * chunk);
        }
        h->fact_row_lo = lo;
    }
    h->emb_rows[which] = hi - lo;
    const size_t n = (size_t)std::max<int64_t>(hi - lo, 1) * dim;
    HRAG_CUDA(cudaMalloc(&h->emb_hi[which], n * 2));
    HRAG_CUDA(cudaMalloc(&h->emb_lo[which], n * 2));
    return 0;
}

int hrag_load_embeddings_chunk(hrag_t* h, int which, int64_t row0, int64_t n_rows, const float* emb, int on_device) {
    HRAG_CHECK(h && (which == 0 || which == 1) && emb, "hrag_load_embeddings_chunk: bad arguments");
    HRAG_CHECK(h->emb_hi[which] != nullptr && h->emb[which] == nullptr,
               "hrag_load_embeddings_chunk: call hrag_load_embeddings_begin first");
    HRAG_CUDA(cudaSetDevice(h->device));
    const int64_t lo = which == 0 ? h->fact_row_lo : 0, hi = lo + h->emb_rows[which];
    const int64_t total = which == 0 ? h->n_facts_global : h->emb_rows[1];
    HRAG_CHECK(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= total, "hrag_load_embeddings_chunk: rows out of range");
    const int64_t a = std::max(row0, lo), b = std::min(row0 + n_rows, hi);      // the part this handle keeps
    if (a >= b) return 0;
    const size_t n = (size_t)(b - a) * h->dim;
    const float* src = emb + (size_t)(a - row0) * h->dim;
    if (!on_device) {
        HRAG_TRY(h->d_reset.ensure(n * sizeof(float)));                          // staging
        HRAG_CUDA(cudaMemcpyAsync(h->d_reset.p, src, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        src = h->d_reset.as<float>();
    }
    HRAG_TRY(split_bf16(src, (int64_t)n, static_cast<char*>(h->emb_hi[which]) + (size_t)(a - lo) * h->dim * 2,
                        static_cast<char*>(h->emb_lo[which]) + (size_t)(a - lo) * h->dim * 2, h->stream));
    HRAG_CUDA(cudaStreamSynchronize(h->stream));
    return 0;
}

int hrag_set_options(hrag_t* h, int ppr_method, int ppr_iters, int ppr_batch, int sim_mode) {
    HRAG_CHECK(h, "hrag_set_options: null handle");
    h->graph_generation += 1;
    if (ppr_method >= 0) {
        HRAG_CHECK(ppr_method == HRAG_PPR_POWER || ppr_method == HRAG_PPR_CHEBYSHEV, "bad ppr_method");
        h->ppr_method = ppr_method;
    }
    if (ppr_iters > 0) h->ppr_iters = ppr_iters;
    if (ppr_batch > 0) {
        HRAG_CHECK(ppr_batch <= 64, "ppr_batch must be <= 64");
        h->ppr_batch = ppr_batch;
    }
    if (sim_mode >= 0) {
        HRAG_CHECK(sim_mode == HRAG_SIM_FP32 || sim_mode == HRAG_SIM_BF16X3 || sim_mode == HRAG_SIM_BF16,
                   "bad sim_mode");
        h->sim_mode = sim_mode;
    }
    return 0;
}

int hrag_set_ppr_precision(hrag_t* h, int precision, int sweeps1, int sweeps2) {
    HRAG_CHECK(h, "hrag_set_ppr_precision: null handle");
    if (precision >= 0) {
        HRAG_CHECK(precision == HRAG_PPR_FP32 || precision == HRAG_PPR_MIXED, "bad ppr precision");
        h->ppr_precision = precision;
    }
    if (sweeps1 > 0) h->mixed_m1 = sweeps1;
    if (sweeps2 > 0) h->mixed_m2 = sweeps2;
    return 0;
}

int hrag_stage_a(hrag_t* h, int32_t B, const float* q_fact, int32_t k, int32_t* top_idx, float* top_score,
                 int32_t* n_valid) {
    HRAG_CHECK(h && q_fact && top_idx && top_score && n_valid, "hrag_stage_a: null argument");
    HRAG_CHECK(B >= 0 && k >= 1 && k <= kMaxKeptFacts, "hrag_stage_a: k (linking_top_k) must be in [1, 32]");
    HRAG_CHECK(h->dim > 0, "hrag_stage_a: embeddings not loaded");
    HRAG_CUDA(cudaSetDevice(h->device));
    const int64_t chunk = chunk_a(h, k);
    HRAG_TRY(h->d_q.ensure((size_t)std::min<int64_t>(chunk, B) * h->dim * sizeof(float)));
    HRAG_TRY(h->d_top_idx.ensure((size_t)std::max(B, 1) * k * sizeof(int)));
    HRAG_TRY(h->d_top_score.ensure((size_t)std::max(B, 1) * k * sizeof(float)));
    HRAG_TRY(h->d_nvalid.ensure((size_t)std::max(B, 1) * sizeof(int)));
    for (int64_t q0 = 0; q0 < B; q0 += chunk) {
        const int nb = (int)std::min<int64_t>(chunk, B - q0);
        HRAG_TRY(h2d(h, h->d_q.p, q_fact + (size_t)q0 * h->dim, (size_t)nb * h->dim * sizeof(float)));
        HRAG_TRY(dev_stage_a(h, nb, h->d_q.as<float>(), k, h->d_top_idx.as<int>() + q0 * k,
                             h->d_top_score.as<float>() + q0 * k, h->d_nvalid.as<int>() + q0));
    }
    if (B > 0) {
        HRAG_TRY(d2h(h, top_idx, h->d_top_idx.p, (size_t)B * k * sizeof(int)));
        HRAG_TRY(d2h(h, top_score, h->d_top_score.p, (size_t)B * k * sizeof(float)));
        HRAG_TRY(d2h(h, n_valid, h->d_nvalid.p, (size_t)B * sizeof(int)));
    }
    return resolve_spans(h);
}

// tables, graph and embeddings must describe the same index (a passage matrix with more rows than passage_vid
// would make the similarity kernel write past the score buffer)
static int check_loaded(hrag_t* h, const char* who, bool need_facts) {
    HRAG_CHECK(h->dim > 0 && h->g.n_global > 0 && h->t.passage_vid, std::string(who) + ": graph/tables/embeddings not loaded");
    HRAG_CHECK(h->emb_rows[1] == h->t.n_passages,
               std::string(who) + ": passage embeddings have " + std::to_string(h->emb_rows[1]) + " rows but passage_vid has " +
                   std::to_string(h->t.n_passages));
    HRAG_CHECK(!need_facts || h->n_facts_global == 0 || h->n_facts_global == h->t.n_facts,
               std::string(who) + ": fact embeddings have " + std::to_string(h->n_facts_global) + " rows but the fact tables have " +
                   std::to_string(h->t.n_facts));
    return 0;
}

int hrag_stage_b(hrag_t* h, int32_t B, const float* q_pass, const int32_t* kept_fact_idx,
                 const float* kept_fact_score, int32_t k_facts, const uint8_t* dpr_only, float damping,
                 float passage_node_weight, int32_t link_top_k, int32_t topk, int32_t iters, float tol,
                 int32_t* out_ids, float* out_scores) {
    HRAG_CHECK(h && q_pass && out_ids && out_scores, "hrag_stage_b: null argument");
    HRAG_CHECK(k_facts == 0 || (kept_fact_idx && kept_fact_score), "hrag_stage_b: kept facts missing");
    HRAG_CHECK(B >= 0 && k_facts >= 0 && k_facts <= kMaxKeptFacts && topk >= 1 && topk <= 2048,
               "hrag_stage_b: bad sizes (at most 32 kept facts per query, topk <= 2048)");
    HRAG_CHECK(damping > 0.f && damping < 1.f, "hrag_stage_b: damping must be in (0, 1)");
    HRAG_CHECK(iters >= 0 && tol >= 0.f, "hrag_stage_b: iters and tol must be >= 0 (0 = derive from damping)");
    HRAG_TRY(check_loaded(h, "hrag_stage_b", k_facts > 0));
    HRAG_CUDA(cudaSetDevice(h->device));
    const int64_t chunk = chunk_b(h);
    const int kf = std::max(k_facts, 1);
    HRAG_TRY(h->d_q2.ensure((size_t)std::min<int64_t>(chunk, std::max(B, 1)) * h->dim * sizeof(float)));
    HRAG_TRY(h->d_kept_idx.ensure((size_t)std::max(B, 1) * kf * sizeof(int)));
    HRAG_TRY(h->d_kept_score.ensure((size_t)std::max(B, 1) * kf * sizeof(float)));
    HRAG_TRY(h->d_dpr.ensure((size_t)std::max(B, 1)));
    HRAG_TRY(h->d_out_ids.ensure((size_t)std::max(B, 1) * topk * sizeof(int)));
    HRAG_TRY(h->d_out_scores.ensure((size_t)std::max(B, 1) * topk * sizeof(float)));
    if (B == 0) return resolve_spans(h);
    if (k_facts > 0) {
        HRAG_TRY(h2d(h, h->d_kept_idx.p, kept_fact_idx, (size_t)B * k_facts * sizeof(int)));
        HRAG_TRY(h2d(h, h->d_kept_score.p, kept_fact_score, (size_t)B * k_facts * sizeof(float)));
    }
    if (dpr_only) HRAG_TRY(h2d(h, h->d_dpr.p, dpr_only, (size_t)B));
    for (int64_t q0 = 0; q0 < B; q0 += chunk) {
        const int nb = (int)std::min<int64_t>(chunk, B - q0);
        HRAG_TRY(h2d(h, h->d_q2.p, q_pass + (size_t)q0 * h->dim, (size_t)nb * h->dim * sizeof(float)));
        HRAG_TRY(dev_stage_b(h, nb, h->d_q2.as<float>(), h->d_kept_idx.as<int>() + q0 * k_facts,
                             h->d_kept_score.as<float>() + q0 * k_facts, k_facts,
                             dpr_only ? h->d_dpr.as<uint8_t>() + q0 : nullptr, damping, passage_node_weight,
                             link_top_k, topk, iters, tol, h->d_out_ids.as<int>() + q0 * topk,
                             h->d_out_scores.as<float>() + q0 * topk));
    }
    HRAG_TRY(d2h(h, out_ids, h->d_out_ids.p, (size_t)B * topk * sizeof(int)));
    HRAG_TRY(d2h(h, out_scores, h->d_out_scores.p, (size_t)B * topk * sizeof(float)));
    return resolve_spans(h);
}

int hrag_retrieve_resident(hrag_t* h, int32_t B, const float* d_q_fact, const float* d_q_pass, float damping,
                           float passage_node_weight, int32_t link_top_k, int32_t topk, int32_t iters, float tol,
                           int32_t* d_out_ids, float* d_out_scores) {
    HRAG_CHECK(h && d_q_fact && d_q_pass && d_out_ids && d_out_scores, "hrag_retrieve_resident: null argument");
    HRAG_CHECK(B >= 0 && link_top_k >= 1 && link_top_k <= kMaxKeptFacts && topk >= 1 && topk <= 2048,
               "hrag_retrieve_resident: bad sizes (linking_top_k in [1, 32], topk <= 2048)");
    HRAG_CHECK(damping > 0.f && damping < 1.f, "hrag_retrieve_resident: damping must be in (0, 1)");
    HRAG_CHECK(iters >= 0 && tol >= 0.f, "hrag_retrieve_resident: iters and tol must be >= 0");
    HRAG_TRY(check_loaded(h, "hrag_retrieve_resident", true));
    HRAG_CUDA(cudaSetDevice(h->device));
    const int64_t chunk = std::min(chunk_a(h, link_top_k), chunk_b(h));
    const int k = link_top_k;
    HRAG_TRY(h->d_top_idx.ensure((size_t)chunk * k * sizeof(int)));
    HRAG_TRY(h->d_top_score.ensure((size_t)chunk * k * sizeof(float)));
    HRAG_TRY(h->d_nvalid.ensure((size_t)chunk * sizeof(int)));
    for (int64_t q0 = 0; q0 < B; q0 += chunk) {
        const int nb = (int)std::min<int64_t>(chunk, B - q0);
        HRAG_TRY(dev_stage_a(h, nb, d_q_fact + (size_t)q0 * h->dim, k, h->d_top_idx.as<int>(),
                             h->d_top_score.as<float>(), h->d_nvalid.as<int>()));
        // identity recognition-memory filter: the candidates are the kept facts
        HRAG_TRY(dev_stage_b(h, nb, d_q_pass + (size_t)q0 * h->dim, h->d_top_idx.as<int>(),
                             h->d_top_score.as<float>(), k, nullptr, damping, passage_node_weight, link_top_k,
                             topk, iters, tol, d_out_ids + q0 * topk, d_out_scores + q0 * topk));
    }
    return resolve_spans(h);
}

int hrag_ppr(hrag_t* h, int32_t B, const float* reset, float damping, int32_t iters, float tol, float* out) {
    HRAG_CHECK(h && reset && out, "hrag_ppr: null argument");
    HRAG_CHECK(B >= 0 && damping > 0.f && damping < 1.f, "hrag_ppr: bad arguments");
    HRAG_CHECK(iters >= 0 && tol >= 0.f, "hrag_ppr: iters and tol must be >= 0 (0 = derive from damping)");
    HRAG_CHECK(h->g.n_global > 0, "hrag_ppr: graph not loaded");
    HRAG_CUDA(cudaSetDevice(h->device));
    const int N = h->g.n_global;
    // same gate as stage B: batches of <= 16 reset vectors run the fp32 solver at their own width
    const SweepPlan plan = plan_sweeps(h, damping, iters, tol, h->ppr_precision == HRAG_PPR_MIXED && B > 16);
    const bool mixed = plan.mixed;
    const int Bp = mixed ? 32 : round_batch(std::min(h->ppr_batch, std::max(B, 1)));
    if (mixed) { HRAG_TRY(ensure_state_mixed(h)); HRAG_TRY(h->V.ensure(state_rows(h) * 32 * sizeof(float))); }
    else HRAG_TRY(ensure_state(h, Bp));
    if (mixed && plan.check) { h->check_tol = plan.tol; h->check_kappa = plan.kappa; }
    HRAG_TRY(h->d_reset.ensure((size_t)Bp * N * sizeof(float)));
    HRAG_TRY(h->d_scores.ensure((size_t)Bp * N * sizeof(float)));
    for (int q0 = 0; q0 < B; q0 += Bp) {
        const int nb = std::min(Bp, B - q0);
        HRAG_TRY(h2d(h, h->d_reset.p, reset + (size_t)q0 * N, (size_t)nb * N * sizeof(float)));
        HRAG_TRY(reset_to_state(h->d_reset.as<float>(), nb, N, Bp, h->V.as<float>(), h->stream));
        if (mixed) {
            void *X0 = nullptr, *D = nullptr;
            double* vsum = h->sums.as<double>() + kSumV;
            HRAG_TRY(mixed_prepare_rhs(h->V.as<float>(), (int64_t)N, damping, h->partials.as<float>(), vsum,
                                       h->mixed_aux.as<float>(), h->H[0].p, h->stream));
            HRAG_TRY(dev_ppr_mixed(h, plan, damping, nullptr, h->V.as<float>(), h->H[0].p, h->H[0].p,
                                   h->mixed_aux.as<float>(), vsum, &X0, &D));
            HRAG_TRY(state_to_scores_mixed(X0, D, 1.f / kMixedT, nb, N, h->sums.as<double>(),
                                           h->sums.as<double>() + 32, h->d_scores.as<float>(), h->stream));
            HRAG_TRY(p2p_signal(h));
        } else {
            float* Z = nullptr;
            HRAG_TRY(dev_ppr(h, Bp, plan.iters, damping, &Z));
            HRAG_TRY(state_to_scores(Z, nb, N, Bp, h->sums.as<double>(), h->d_scores.as<float>(), h->stream));
        }
        HRAG_TRY(d2h(h, out + (size_t)q0 * N, h->d_scores.p, (size_t)nb * N * sizeof(float)));
        HRAG_CUDA(cudaStreamSynchronize(h->stream));
    }
    return resolve_spans(h);
}

int hrag_similarity(hrag_t* h, int which, int32_t B, const float* q, float* out) {
    HRAG_CHECK(h && q && out && (which == 0 || which == 1), "hrag_similarity: bad arguments");
    HRAG_CHECK(h->dim > 0 && h->emb_rows[which] > 0, "hrag_similarity: embeddings not loaded");
    HRAG_CUDA(cudaSetDevice(h->device));
    const int64_t M = h->emb_rows[which], ld = pad4(M);
    const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>((int64_t)(2e9 / (4.0 * (double)ld)), 1024));
    hrag::Buf& Sb = which == 0 ? h->S_fact : h->S_pass;
    hrag::Buf& mm = which == 0 ? h->mm_fact : h->mm_pass;
    HRAG_TRY(Sb.ensure((size_t)std::min<int64_t>(chunk, std::max(B, 1)) * ld * sizeof(float)));
    HRAG_TRY(mm.ensure((size_t)std::min<int64_t>(chunk, std::max(B, 1)) * sizeof(float2)));
    HRAG_TRY(h->d_q.ensure((size_t)std::min<int64_t>(chunk, std::max(B, 1)) * h->dim * sizeof(float)));
    for (int64_t q0 = 0; q0 < B; q0 += chunk) {
        const int nb = (int)std::min<int64_t>(chunk, B - q0);
        HRAG_TRY(h2d(h, h->d_q.p, q + (size_t)q0 * h->dim, (size_t)nb * h->dim * sizeof(float)));
        HRAG_TRY(sim_dispatch(h, h->d_q.as<float>(), nb, which, Sb.as<float>(), ld));
        HRAG_TRY(row_minmax_topk(Sb.as<float>(), nb, M, ld, 0, mm.as<float2>(), nullptr, nullptr, nullptr, h->stream));
        HRAG_TRY(minmax_apply(Sb.as<float>(), nb, M, ld, mm.as<float2>(), h->stream));
        HRAG_CUDA(cudaMemcpy2DAsync(out + (size_t)q0 * M, (size_t)M * sizeof(float), Sb.p, (size_t)ld * sizeof(float),
                                    (size_t)M * sizeof(float), (size_t)nb, cudaMemcpyDeviceToHost, h->stream));
        h->stats.d2h_bytes += (int64_t)nb * M * 4;
        HRAG_CUDA(cudaStreamSynchronize(h->stream));
    }
    (which == 0 ? h->last_fact_rows : h->last_pass_rows) = 0;
    return resolve_spans(h);
}

int hrag_topk_similarity(hrag_t* h, int which, int32_t B, const float* q, int32_t k, int32_t* out_ids,
                         float* out_scores) {
    HRAG_CHECK(h && q && out_ids && out_scores && (which == 0 || which == 1), "hrag_topk_similarity: bad arguments");
    HRAG_CHECK(k >= 1 && k <= 2048 && B >= 0, "hrag_topk_similarity: k must be in [1, 2048]");
    HRAG_CHECK(h->dim > 0 && h->emb_rows[which] > 0, "hrag_topk_similarity: embeddings not loaded");
    HRAG_CUDA(cudaSetDevice(h->device));
    const int64_t M = h->emb_rows[which], ld = pad4(M);
    const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>((int64_t)(4e9 / (4.0 * (double)ld)), 1024));
    hrag::Buf& Sb = which == 0 ? h->S_fact : h->S_pass;
    const int64_t cb = std::min<int64_t>(chunk, std::max(B, 1));
    HRAG_TRY(Sb.ensure((size_t)cb * ld * sizeof(float)));
    HRAG_TRY(h->d_q.ensure((size_t)cb * h->dim * sizeof(float)));
    HRAG_TRY(h->d_out_ids.ensure((size_t)cb * k * sizeof(int)));
    HRAG_TRY(h->d_out_scores.ensure((size_t)cb * k * sizeof(float)));
    for (int64_t q0 = 0; q0 < B; q0 += chunk) {
        const int nb = (int)std::min<int64_t>(chunk, B - q0);
        HRAG_TRY(h2d(h, h->d_q.p, q + (size_t)q0 * h->dim, (size_t)nb * h->dim * sizeof(float)));
        {
            StageTimer tm(h, which == 0 ? ST_SIM_FACT : ST_SIM_PASS);
            HRAG_TRY(sim_dispatch(h, h->d_q.as<float>(), nb, which, Sb.as<float>(), ld));
        }
        {
            StageTimer tm(h, ST_TOPK);
            HRAG_TRY(row_topk(Sb.as<float>(), nb, M, ld, k, h->d_out_ids.as<int>(), h->d_out_scores.as<float>(), h->stream));
        }
        HRAG_TRY(d2h(h, out_ids + (size_t)q0 * k, h->d_out_ids.p, (size_t)nb * k * sizeof(int)));
        HRAG_TRY(d2h(h, out_scores + (size_t)q0 * k, h->d_out_scores.p, (size_t)nb * k * sizeof(float)));
        HRAG_CUDA(cudaStreamSynchronize(h->stream));
    }
    (which == 0 ? h->last_fact_rows : h->last_pass_rows) = 0;
    return resolve_spans(h);
}

int hrag_knn_threshold(hrag_t* h, int which, int32_t B, const float* q, float min_score, int32_t kmax,
                       int32_t* out_ids, float* out_scores, int32_t* n_found) {
    HRAG_CHECK(h && q && out_ids && out_scores && n_found && (which == 0 || which == 1), "hrag_knn_threshold: bad arguments");
    HRAG_CHECK(kmax >= 1 && kmax <= kCandidateCap && B >= 0, "hrag_knn_threshold: kmax must be in [1, 512]");
    HRAG_CHECK(h->dim > 0 && h->emb_rows[which] > 0 && h->emb_hi[which] != nullptr,
               "hrag_knn_threshold: embeddings not loaded (needs the tensor-core layout: dim % 8 == 0)");
    HRAG_CHECK(h->sim_mode != HRAG_SIM_FP32, "hrag_knn_threshold: the threshold epilogue lives in the tcgen05 kernel");
    HRAG_CUDA(cudaSetDevice(h->device));
    const int64_t M = h->emb_rows[which];
    const int64_t chunk = 1024;
    const int64_t cb = std::min<int64_t>(chunk, std::max(B, 1));
    HRAG_TRY(h->d_q.ensure((size_t)cb * h->dim * sizeof(float)));
    HRAG_TRY(h->q_hi.ensure((size_t)cb * h->dim * 2));
    HRAG_TRY(h->q_lo.ensure((size_t)cb * h->dim * 2));
    HRAG_TRY(h->part_keys.ensure((size_t)cb * kCandidateCap * sizeof(uint64_t)));
    HRAG_TRY(h->d_nvalid.ensure((size_t)cb * 2 * sizeof(int)));
    HRAG_TRY(h->d_out_ids.ensure((size_t)cb * kmax * sizeof(int)));
    HRAG_TRY(h->d_out_scores.ensure((size_t)cb * kmax * sizeof(float)));
    int* d_count = h->d_nvalid.as<int>();
    int* d_found = d_count + cb;
    for (int64_t q0 = 0; q0 < B; q0 += chunk) {
        const int nb = (int)std::min<int64_t>(chunk, B - q0);
        HRAG_TRY(h2d(h, h->d_q.p, q + (size_t)q0 * h->dim, (size_t)nb * h->dim * sizeof(float)));
        HRAG_CUDA(cudaMemsetAsync(d_count, 0, (size_t)nb * sizeof(int), h->stream));
        {
            StageTimer tm(h, which == 0 ? ST_SIM_FACT : ST_SIM_PASS);
            HRAG_TRY(split_bf16(h->d_q.as<float>(), (int64_t)nb * h->dim, h->q_hi.p, h->q_lo.p, h->stream));
            HRAG_TRY(sim_tc_threshold(h->q_hi.p, h->q_lo.p, nb, h->emb_hi[which], h->emb_lo[which], M, h->dim,
                                      h->sim_mode == HRAG_SIM_BF16X3 ? 4 : 1, min_score, h->part_keys.as<uint64_t>(),
                                      d_count, kCandidateCap, h->num_sms, h->stream));
        }
        {
            StageTimer tm(h, ST_TOPK);
            HRAG_TRY(sort_candidates(h->part_keys.as<uint64_t>(), d_count, nb, kCandidateCap, kmax, h->d_out_ids.as<int>(),
                                     h->d_out_scores.as<float>(), d_found, h->stream));
        }
        HRAG_TRY(d2h(h, out_ids + (size_t)q0 * kmax, h->d_out_ids.p, (size_t)nb * kmax * sizeof(int)));
        HRAG_TRY(d2h(h, out_scores + (size_t)q0 * kmax, h->d_out_scores.p, (size_t)nb * kmax * sizeof(float)));
        HRAG_TRY(d2h(h, n_found + q0, d_found, (size_t)nb * sizeof(int)));
        HRAG_CUDA(cudaStreamSynchronize(h->stream));
    }
    return resolve_spans(h);
}

int hrag_bench_sweep(hrag_t* h, int32_t B, int32_t sweeps, int32_t method, float* ms_per_sweep) {
    HRAG_CHECK(h && ms_per_sweep && sweeps >= 1, "hrag_bench_sweep: bad arguments");
    HRAG_CHECK(B == 4 || B == 8 || B == 16 || B == 32 || B == 64, "hrag_bench_sweep: B in {4,8,16,32,64}");
    HRAG_CHECK(h->g.n_global > 0, "hrag_bench_sweep: graph not loaded");
    HRAG_CUDA(cudaSetDevice(h->device));
    if (method == 2 || method == 3) {   // fp16-state sweep (Chebyshev form), B = 32; 2 = dense rhs, 3 = compact rhs
        HRAG_CHECK(B == 32, "hrag_bench_sweep: the mixed solver runs at B = 32");
        HRAG_TRY(ensure_state_mixed(h));
        const int* slot_map = nullptr;
        const void* rhs = h->H[0].p;
        if (method == 3) {
            HRAG_CHECK(h->t.passage_vid != nullptr, "hrag_bench_sweep: the compact-rhs sweep needs hrag_load_tables");
            HRAG_TRY(ensure_compact_rhs(h));
            slot_map = h->slot_map[0].as<int>();
            rhs = h->R16[0].p;
            HRAG_CUDA(cudaMemsetAsync(h->R16[0].p, 0x2c, h->R16[0].cap, h->stream));
        }
        const size_t hb = (size_t)h->g.n_global * 32 * 2;
        for (int i = 0; i < 3; ++i) HRAG_CUDA(cudaMemsetAsync(h->H[i].p, 0x2c, hb, h->stream));   // 0x2c2c = 0.065
        cudaEvent_t e0, e1;
        HRAG_CUDA(cudaEventCreate(&e0));
        HRAG_CUDA(cudaEventCreate(&e1));
        for (int pass = 0; pass < 2; ++pass) {
            const int n = pass == 0 ? 3 : sweeps;
            if (pass == 1) HRAG_CUDA(cudaEventRecord(e0, h->stream));
            for (int i = 0; i < n; ++i) {
                void* x = (i & 1) ? h->H[2].p : h->H[1].p;
                void* y = (i & 1) ? h->H[1].p : h->H[2].p;
                HRAG_TRY(mixed_sweep_x(h, 0, x, slot_map, rhs, nullptr, nullptr, y, y, 0.5f, 1.07f, 1.f, nullptr, nullptr));
            }
            if (pass == 1) HRAG_CUDA(cudaEventRecord(e1, h->stream));
        }
        HRAG_CUDA(cudaStreamSynchronize(h->stream));
        float ms = 0.f;
        HRAG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        *ms_per_sweep = ms / sweeps;
        return 0;
    }
    HRAG_TRY(ensure_state(h, B));
    const size_t bytes = (size_t)h->g.n_global * B * sizeof(float);
    HRAG_CUDA(cudaMemsetAsync(h->V.p, 0x3c, bytes, h->stream));     // 0x3c3c3c3c = 0.0115f
    HRAG_CUDA(cudaMemsetAsync(h->XA.p, 0x3c, bytes, h->stream));
    HRAG_CUDA(cudaMemsetAsync(h->XC.p, 0x3c, bytes, h->stream));
    float* A = h->XA.as<float>();
    float* C = h->XC.as<float>();
    const float* V = h->V.as<float>();
    cudaEvent_t e0, e1;
    HRAG_CUDA(cudaEventCreate(&e0));
    HRAG_CUDA(cudaEventCreate(&e1));
    for (int pass = 0; pass < 2; ++pass) {   // pass 0 = warm-up (3 sweeps), pass 1 = timed
        const int n = pass == 0 ? 3 : sweeps;
        if (pass == 1) HRAG_CUDA(cudaEventRecord(e0, h->stream));
        for (int i = 0; i < n; ++i) {
            const float* x = (i & 1) ? C : A;
            float* y = (i & 1) ? A : C;
            if (method == HRAG_PPR_CHEBYSHEV) HRAG_TRY(ppr_sweep(h->g, B, x, V, y, y, 0.5f, 1.07f, nullptr, nullptr, h->stream));
            else HRAG_TRY(ppr_sweep(h->g, B, x, V, nullptr, y, 0.5f, 1.f, nullptr, nullptr, h->stream));
            HRAG_TRY(exchange_rows(h, y, B));
        }
        if (pass == 1) HRAG_CUDA(cudaEventRecord(e1, h->stream));
    }
    HRAG_CUDA(cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    HRAG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ms_per_sweep = ms / sweeps;
    for (auto& s : h->spans) { h->pool.push_back(s.a); h->pool.push_back(s.b); }
    h->spans.clear();
    return 0;
}

int hrag_plan_sweeps(float damping, float tol, int32_t iters, int32_t batch, int32_t* use_mixed, int32_t* fp32_sweeps,
                     int32_t* mixed_sweeps1, int32_t* mixed_sweeps2, double* predicted_error) {
    HRAG_CHECK(use_mixed && fp32_sweeps && mixed_sweeps1 && mixed_sweeps2 && predicted_error, "hrag_plan_sweeps: null argument");
    HRAG_CHECK(damping > 0.f && damping < 1.f && tol >= 0.f && iters >= 0, "hrag_plan_sweeps: bad arguments");
    const SweepPlan p = plan_sweeps_raw(HRAG_PPR_CHEBYSHEV, 0, 0, 0, damping, iters, tol, batch > 16);
    const double a = damping, sig = a / (1.0 + std::sqrt(1.0 - a * a)), noise = kHalfNoise / (1.0 - a);
    *use_mixed = p.mixed ? 1 : 0;
    *fp32_sweeps = p.iters;
    *mixed_sweeps1 = p.m1;
    *mixed_sweeps2 = p.m2;
    *predicted_error = p.mixed ? (noise + 2.0 * std::pow(sig, p.m1)) * p.kappa : 2.0 * std::pow(sig, p.iters);
    return 0;
}

int hrag_set_tuning(hrag_t* h, int k5_debug) {
    HRAG_CHECK(h, "hrag_set_tuning: null handle");
    h->graph_generation += 1;
    if (k5_debug >= 0) h->k5_debug = k5_debug;
    return 0;
}

void* hrag_stream(hrag_t* h) { return h ? (void*)h->stream : nullptr; }

int hrag_get_stats(hrag_t* h, hrag_stats_t* out) {
    HRAG_CHECK(h && out, "hrag_get_stats: null argument");
    h->stats.kernel_launches = launches_since_reset();
    h->stats.ppr_residual = h->last_rho;
    h->stats.ppr_error_bound = h->last_bound;
    *out = h->stats;
    return 0;
}

int hrag_reset_stats(hrag_t* h) {
    HRAG_CHECK(h, "hrag_reset_stats: null handle");
    h->stats = hrag_stats_t{};
    reset_launch_counter();
    return 0;
}

int hrag_debug_keep_scores(hrag_t* h, int keep) {
    HRAG_CHECK(h, "hrag_debug_keep_scores: null handle");
    h->keep_fact_scores = keep != 0;
    return 0;
}

int hrag_debug_copy(hrag_t* h, int which, float* host_out, int64_t max_elems, int64_t* n_written) {
    HRAG_CHECK(h && host_out && n_written, "hrag_debug_copy: null argument");
    HRAG_CUDA(cudaSetDevice(h->device));
    const hrag::Buf& b = which == 0 ? h->S_fact : h->S_pass;
    const int64_t rows = which == 0 ? h->last_fact_rows : h->last_pass_rows;
    const int64_t cols = which == 0 ? h->emb_rows[0] : h->t.n_passages;
    const int64_t ld = pad4(cols);
    HRAG_CHECK(rows * cols <= max_elems, "hrag_debug_copy: host buffer too small");
    HRAG_CUDA(cudaStreamSynchronize(h->stream));
    if (rows && cols)
        HRAG_CUDA(cudaMemcpy2D(host_out, (size_t)cols * sizeof(float), b.p, (size_t)ld * sizeof(float),
                               (size_t)cols * sizeof(float), (size_t)rows, cudaMemcpyDeviceToHost));
    *n_written = rows * cols;
    return 0;
}

}  // extern "C"
