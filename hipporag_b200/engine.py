"""Python host side of the B200 retrieval engine: thin, typed wrappers over the C ABI.

``Engine`` mirrors the state ``HippoRAG.prepare_retrieval_objects`` materialises
(``/root/reference/src/hipporag/HippoRAG.py:1287-1389``) -- graph, integer tables, fact and
passage embeddings -- as device-resident arrays, and exposes the two GPU stages that bracket the
recognition-memory (LLM) filter of ``HippoRAG.retrieve`` (``:459-480``):

* stage A = ``get_fact_scores`` + the top-k of ``rerank_facts``          (``:1427-1465, 1683-1688``)
* stage B = ``dense_passage_retrieval`` + ``graph_search_with_fact_entities`` + ``run_ppr``
  + the top-k slice of ``_build_retrieval_result``           (``:1467-1502, 1544-1656, 1709-1749, 501-507``)

``B200Retriever`` is the same path on raw arrays (synthetic configs, no HippoRAG object).
Nothing here computes on the CPU: every numeric step is a call into ``libhrag_b200.so``.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import (HragError, PPR_CHEBYSHEV, PPR_FP32, PPR_MIXED, PPR_POWER, SIM_BF16, SIM_BF16X3,  # noqa: F401
                   SIM_FP32)


def build_transition_csr(n_nodes: int, edge_src, edge_dst, edge_w) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """CSR of P = W D^-1 from an igraph-style undirected multigraph edge list.

    Host-side ingest of the graph ``add_new_edges`` builds (``HippoRAG.py:1189-1223``): every
    edge (u, v, w) contributes w to W[u, v] and W[v, u]; parallel edges sum (the reference emits
    each fact as (s, o) and (o, s), ``:907-910``); edges with w <= 0 carry nothing; columns are
    divided by the vertex strength.  Returns (row_ptr int64, col int32, val float32).
    """
    import scipy.sparse as sp
    src = np.asarray(edge_src, dtype=np.int64)
    dst = np.asarray(edge_dst, dtype=np.int64)
    w = np.asarray(edge_w, dtype=np.float64)
    if src.shape != dst.shape or src.shape != w.shape:
        raise ValueError("edge_src, edge_dst, edge_w must have the same length")
    if src.size and (min(src.min(), dst.min()) < 0 or max(src.max(), dst.max()) >= n_nodes):
        raise ValueError("edge endpoint out of range")
    keep = w > 0
    src, dst, w = src[keep], dst[keep], w[keep]
    W = sp.coo_matrix((np.concatenate([w, w]), (np.concatenate([src, dst]), np.concatenate([dst, src]))),
                      shape=(n_nodes, n_nodes)).tocsr()
    W.sum_duplicates()
    W.sort_indices()
    strength = np.asarray(W.sum(axis=0)).ravel()
    inv = np.zeros_like(strength)
    nz = strength > 0
    inv[nz] = 1.0 / strength[nz]
    val = (W.data * inv[W.indices]).astype(np.float32)
    return W.indptr.astype(np.int64), W.indices.astype(np.int32), val


def plan_sweeps(damping: float = 0.5, tol: float = 0.0, iters: int = 0, batch: int = 32) -> dict:
    """What the library will run for (damping, tol, iters) on a batch of ``batch`` PPR columns (``hrag_plan_sweeps``;
    pure host code, works without a GPU): solver, sweep counts, predicted relative L1 error."""
    lib = _lib.load()
    mixed, it32, m1, m2 = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
    err = C.c_double()
    _lib.check(lib.hrag_plan_sweeps(damping, tol, iters, batch, C.byref(mixed), C.byref(it32), C.byref(m1), C.byref(m2),
                                    C.byref(err)))
    return {"solver": "mixed" if mixed.value else "fp32", "fp32_sweeps": it32.value,
            "mixed_sweeps": (m1.value, 1, m2.value), "predicted_error": err.value}


def shard_rows(n_nodes: int, rank: int, world: int) -> Tuple[int, int]:
    """Node-range partition used by every rank: rows [rank*ceil(N/world), (rank+1)*ceil(N/world))."""
    chunk = -(-n_nodes // world)
    return min(n_nodes, rank * chunk), min(n_nodes, (rank + 1) * chunk)


def balanced_row_bounds(row_ptr, world: int) -> np.ndarray:
    """Work-balanced node-range partition: rank r owns rows [b[r], b[r + 1]) with equal shares of
    cost = non-zeros + 4 per row (a row's epilogue streams cost about four gathers)."""
    row_ptr = np.asarray(row_ptr, dtype=np.int64)
    n = row_ptr.shape[0] - 1
    cost = row_ptr[:-1] + 4 * np.arange(n, dtype=np.int64)          # cost of all rows BEFORE row r
    total = float(row_ptr[-1] + 4 * n)
    b = np.empty(world + 1, dtype=np.int64)
    b[0], b[world] = 0, n
    for k in range(1, world):
        b[k] = int(np.searchsorted(cost, total * k / world, side="left"))
    return np.maximum.accumulate(b)


def slice_csr_rows(row_ptr, col, val, lo: int, hi: int):
    """Rows [lo, hi) of a CSR matrix as a self-contained CSR (columns stay global)."""
    a, b = int(row_ptr[lo]), int(row_ptr[hi])
    return np.ascontiguousarray(row_ptr[lo:hi + 1] - a), col[a:b], val[a:b]


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.int32)


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else C.c_void_p(a.ctypes.data)


class Engine:
    """One handle = one B200.  Not thread-safe (like the reference's ``HippoRAG`` object)."""

    def __init__(self, device: int = 0, shard_mode: int = 0):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        dev = (C.c_int * 1)(device)
        _lib.check(self._lib.hrag_create(dev, 1, shard_mode, C.byref(self._h)))
        self.device = device
        self.rank, self.world = 0, 1
        self.n_nodes = 0
        self.n_passages = 0
        self.n_facts = 0
        self.dim = 0
        self._keep = []          # device tensors the handle borrows

    # ---------------------------------------------------------------- lifecycle
    def close(self):
        if self._h:
            self._lib.hrag_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---------------------------------------------------------------- multi-GPU
    @staticmethod
    def new_comm_id() -> bytes:
        buf = C.create_string_buffer(128)
        _lib.check(_lib.load().hrag_comm_unique_id(buf))
        return buf.raw

    def init_comm(self, comm_id: bytes, rank: int, world: int):
        buf = C.create_string_buffer(comm_id, 128)
        _lib.check(self._lib.hrag_comm_init(self._h, buf, rank, world))
        self.rank, self.world = rank, world

    def p2p_export(self) -> bytes:
        """64-byte CUDA IPC handle of this rank's PPR state (after init_comm + load_graph)."""
        buf = C.create_string_buffer(64)
        _lib.check(self._lib.hrag_p2p_export(self._h, buf))
        return buf.raw

    def p2p_import(self, handles: Sequence[bytes]):
        """Handles of all ranks in rank order -> fused sweep + exchange (peer stores over NVLink)."""
        blob = C.create_string_buffer(b"".join(handles), 64 * len(handles))
        _lib.check(self._lib.hrag_p2p_import(self._h, blob, len(handles)))

    # ---------------------------------------------------------------- uploads
    def load_graph(self, n_nodes: int, edge_src, edge_dst, edge_w):
        """igraph-style edge list -> device CSR of P (built by the library: hrag_load_graph_coo)."""
        s, d = _i32(edge_src), _i32(edge_dst)
        w = np.ascontiguousarray(edge_w, dtype=np.float64)
        if s.shape != d.shape or s.shape != w.shape:
            raise ValueError("edge_src, edge_dst, edge_w must have the same length")
        _lib.check(self._lib.hrag_load_graph_coo(self._h, n_nodes, int(s.shape[0]), _ptr(s), _ptr(d), _ptr(w)))
        self.n_nodes = n_nodes

    def load_graph_csr(self, n_nodes: int, row_ptr, col, val, balanced: bool = True):
        """Full CSR of P; with node-range sharding this rank's row slice is cut out here -- by default along a
        work-balanced partition (``balanced_row_bounds``), ``balanced=False`` = equal row counts (``shard_rows``)."""
        row_ptr = np.ascontiguousarray(row_ptr, dtype=np.int64)
        col, val = _i32(col), _f32(val)
        lo, hi = (0, n_nodes)
        if self.world > 1:
            if balanced:
                bounds = np.ascontiguousarray(balanced_row_bounds(row_ptr, self.world), dtype=np.int64)
                _lib.check(self._lib.hrag_comm_set_row_bounds(self._h, _ptr(bounds), self.world))
                lo, hi = int(bounds[self.rank]), int(bounds[self.rank + 1])
            else:
                lo, hi = shard_rows(n_nodes, self.rank, self.world)
            row_ptr, col, val = slice_csr_rows(row_ptr, col, val, lo, hi)
        _lib.check(self._lib.hrag_load_graph_csr(self._h, n_nodes, lo, hi, int(col.shape[0]), _ptr(row_ptr),
                                                 _ptr(col), _ptr(val)))
        self.n_nodes = n_nodes

    def load_tables(self, passage_vid, fact_subj_vid, fact_obj_vid, ent_chunk_count):
        pv, fs, fo, cc = _i32(passage_vid), _i32(fact_subj_vid), _i32(fact_obj_vid), _i32(ent_chunk_count)
        if fs.shape != fo.shape:
            raise ValueError("fact_subj_vid / fact_obj_vid length mismatch")
        if cc.shape[0] != self.n_nodes:
            raise ValueError("ent_chunk_count must have one entry per vertex")
        _lib.check(self._lib.hrag_load_tables(self._h, pv.shape[0], _ptr(pv), fs.shape[0], _ptr(fs), _ptr(fo),
                                              _ptr(cc)))
        self.n_passages, self.n_facts = int(pv.shape[0]), int(fs.shape[0])

    def load_embeddings(self, fact_emb, passage_emb):
        """[F, d] and [P, d] fp32; numpy arrays are copied, CUDA torch tensors are borrowed."""
        for which, emb in ((0, fact_emb), (1, passage_emb)):
            if hasattr(emb, "is_cuda"):      # torch tensor already in HBM
                if not (emb.is_cuda and emb.is_contiguous() and str(emb.dtype) == "torch.float32"):
                    raise ValueError("device embeddings must be contiguous fp32 CUDA tensors")
                rows, dim = (int(emb.shape[0]), int(emb.shape[1])) if emb.dim() == 2 else (0, self.dim or 4)
                _lib.check(self._lib.hrag_load_embeddings(self._h, which, rows, dim, C.c_void_p(emb.data_ptr()), 1))
                self._keep.append(emb)
            else:
                emb = _f32(emb)
                if emb.ndim != 2:
                    emb = emb.reshape(0, self.dim or 4)
                rows, dim = emb.shape
                _lib.check(self._lib.hrag_load_embeddings(self._h, which, rows, dim, _ptr(emb), 0))
            self.dim = dim
            if which == 0:
                self.n_facts = int(rows)

    def load_embeddings_streamed(self, which: int, rows: int, dim: int, chunks):
        """Upload [rows, dim] fp32 embeddings chunk by chunk without ever holding them in fp32 on the device:
        ``chunks`` yields (row0, array) with ``array`` a numpy array or a contiguous fp32 CUDA torch tensor."""
        _lib.check(self._lib.hrag_load_embeddings_begin(self._h, which, rows, dim))
        for row0, emb in chunks:
            if hasattr(emb, "is_cuda"):
                if not (emb.is_cuda and emb.is_contiguous() and str(emb.dtype) == "torch.float32"):
                    raise ValueError("device chunks must be contiguous fp32 CUDA tensors")
                _lib.check(self._lib.hrag_load_embeddings_chunk(self._h, which, int(row0), int(emb.shape[0]),
                                                                C.c_void_p(emb.data_ptr()), 1))
            else:
                emb = _f32(emb)
                _lib.check(self._lib.hrag_load_embeddings_chunk(self._h, which, int(row0), int(emb.shape[0]),
                                                                _ptr(emb), 0))
        self.dim = dim
        if which == 0:
            self.n_facts = int(rows)

    def set_options(self, ppr_method: Optional[int] = None, ppr_iters: Optional[int] = None,
                    ppr_batch: Optional[int] = None, sim_mode: Optional[int] = None,
                    ppr_precision: Optional[int] = None, mixed_sweeps: Optional[Tuple[int, int]] = None):
        if ppr_precision is not None or mixed_sweeps is not None:
            m1, m2 = mixed_sweeps or (0, 0)
            _lib.check(self._lib.hrag_set_ppr_precision(self._h, -1 if ppr_precision is None else ppr_precision,
                                                        m1, m2))
        _lib.check(self._lib.hrag_set_options(self._h, -1 if ppr_method is None else ppr_method,
                                              -1 if ppr_iters is None else ppr_iters,
                                              -1 if ppr_batch is None else ppr_batch,
                                              -1 if sim_mode is None else sim_mode))

    # ---------------------------------------------------------------- the two GPU stages
    def stage_a(self, q_fact, k: int = 5):
        """-> (top_idx [B,k] int32, top_score [B,k] fp32 min-maxed, n_valid [B] int32)."""
        q = _f32(q_fact)
        B = q.shape[0]
        idx = np.empty((B, k), dtype=np.int32)
        score = np.empty((B, k), dtype=np.float32)
        nv = np.empty(B, dtype=np.int32)
        _lib.check(self._lib.hrag_stage_a(self._h, B, _ptr(q), k, _ptr(idx), _ptr(score), _ptr(nv)))
        return idx, score, nv

    def stage_b(self, q_pass, kept_idx, kept_score, dpr_only=None, damping: float = 0.5,
                passage_node_weight: float = 0.05, link_top_k: int = 5, topk: int = 200,
                iters: int = 0, tol: float = 0.0):
        """-> (ids [B,topk] int32 into passage order, scores [B,topk] fp32), best first.

        ``tol`` = relative L1 accuracy of each PPR vector (0 = 1e-6); the sweep counts follow from
        ``damping`` and ``tol`` unless ``iters`` pins them (``include/hrag_b200.h``)."""
        q = _f32(q_pass)
        B = q.shape[0]
        kept_idx, kept_score = _i32(kept_idx), _f32(kept_score)
        kf = kept_idx.shape[1] if kept_idx.ndim == 2 else (kept_idx.size // B if B else 0)
        if kf == 0:
            kept_idx = kept_score = None
        if kf and (kept_idx.size != B * kf or kept_score.size != B * kf):
            raise ValueError("kept_idx / kept_score must be [B, k]")
        flags = None if dpr_only is None else np.ascontiguousarray(dpr_only, dtype=np.uint8)
        ids = np.empty((B, topk), dtype=np.int32)
        scores = np.empty((B, topk), dtype=np.float32)
        _lib.check(self._lib.hrag_stage_b(self._h, B, _ptr(q), _ptr(kept_idx), _ptr(kept_score), kf, _ptr(flags),
                                          damping, passage_node_weight, link_top_k or 0, topk, int(iters),
                                          float(tol), _ptr(ids), _ptr(scores)))
        return ids, scores

    def retrieve_resident(self, d_q_fact, d_q_pass, d_out_ids, d_out_scores, damping: float = 0.5,
                          passage_node_weight: float = 0.05, link_top_k: int = 5, topk: int = 200,
                          iters: int = 0, tol: float = 0.0):
        """Whole path on CUDA torch tensors (identity filter); results land in d_out_*."""
        B = int(d_q_fact.shape[0])
        _lib.check(self._lib.hrag_retrieve_resident(
            self._h, B, C.c_void_p(d_q_fact.data_ptr()), C.c_void_p(d_q_pass.data_ptr()), damping,
            passage_node_weight, link_top_k, topk, int(iters), float(tol), C.c_void_p(d_out_ids.data_ptr()),
            C.c_void_p(d_out_scores.data_ptr())))

    def ppr(self, reset, damping: float = 0.5, iters: int = 0, tol: float = 0.0) -> np.ndarray:
        """``run_ppr``'s numeric core: reset [B, N] (or [N]) -> probabilities, same shape."""
        r = _f32(reset)
        single = r.ndim == 1
        r = r.reshape(1, -1) if single else r
        if r.shape[1] != self.n_nodes:
            raise ValueError("reset must have one entry per vertex")
        out = np.empty_like(r)
        _lib.check(self._lib.hrag_ppr(self._h, r.shape[0], _ptr(r), damping, int(iters), float(tol), _ptr(out)))
        return out[0] if single else out

    def similarity(self, which: int, q) -> np.ndarray:
        """Min-max-normalised scores of every fact (which=0) / passage (which=1): [B, rows] fp32."""
        q = _f32(q)
        rows = self.n_facts if which == 0 else self.n_passages
        out = np.empty((q.shape[0], rows), dtype=np.float32)
        _lib.check(self._lib.hrag_similarity(self._h, which, q.shape[0], _ptr(q), _ptr(out)))
        return out

    def topk_similarity(self, which: int, q, k: int):
        """Top-k raw dot products against the fact (0) / passage (1) embedding matrix: (ids, scores) [B, k]."""
        q = _f32(q)
        ids = np.empty((q.shape[0], k), dtype=np.int32)
        scores = np.empty((q.shape[0], k), dtype=np.float32)
        _lib.check(self._lib.hrag_topk_similarity(self._h, which, q.shape[0], _ptr(q), k, _ptr(ids), _ptr(scores)))
        return ids, scores

    def knn_threshold(self, which: int, q, min_score: float, kmax: int = 128):
        """Rows of embedding matrix ``which`` with dot product >= min_score, best first, at most kmax per query:
        (ids [B, kmax] (-1 padded), scores [B, kmax], n_found [B]); selection fused into the GEMM epilogue."""
        q = _f32(q)
        ids = np.empty((q.shape[0], kmax), dtype=np.int32)
        scores = np.empty((q.shape[0], kmax), dtype=np.float32)
        found = np.empty(q.shape[0], dtype=np.int32)
        _lib.check(self._lib.hrag_knn_threshold(self._h, which, q.shape[0], _ptr(q), float(min_score), kmax, _ptr(ids),
                                                _ptr(scores), _ptr(found)))
        return ids, scores, found

    def set_tuning(self, k5_debug: int = -1):
        """Profiling switches of the fused multi-GPU exchange (hrag_set_tuning; -1 keeps the current value)."""
        _lib.check(self._lib.hrag_set_tuning(self._h, k5_debug))

    def bench_sweep(self, batch: int, sweeps: int = 20, method: int = PPR_POWER) -> float:
        ms = C.c_float()
        _lib.check(self._lib.hrag_bench_sweep(self._h, batch, sweeps, method, C.byref(ms)))
        return float(ms.value)

    # ---------------------------------------------------------------- introspection
    @property
    def stream_ptr(self) -> int:
        """cudaStream_t of the handle (wrap with torch.cuda.ExternalStream to record events on it)."""
        return int(self._lib.hrag_stream(self._h) or 0)

    def stats(self) -> dict:
        s = _lib.Stats()
        _lib.check(self._lib.hrag_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    def reset_stats(self):
        _lib.check(self._lib.hrag_reset_stats(self._h))

    def debug_keep_scores(self, keep: bool = True):
        """Make stage A write the raw fact score matrix (tests); the default tensor-core epilogue is fused."""
        _lib.check(self._lib.hrag_debug_keep_scores(self._h, 1 if keep else 0))

    def debug_scores(self, which: int) -> np.ndarray:
        cols = self.n_facts if which == 0 else self.n_passages
        buf = np.empty(1024 * max(cols, 1), dtype=np.float32)
        n = C.c_int64()
        _lib.check(self._lib.hrag_debug_copy(self._h, which, _ptr(buf), buf.shape[0], C.byref(n)))
        return buf[:n.value].reshape(-1, cols) if cols else buf[:0]


FactFilter = Callable[[int, Sequence[int], Sequence[float]], Sequence[int]]


class B200Retriever:
    """The hot path on raw arrays: graph edge list + tables + embeddings in, top-k passages out.

    ``fact_filter(q, fact_idx, fact_score) -> kept positions`` stands in for the recognition
    memory filter (``rerank.py:108``); ``None`` = identity (what every benchmark uses).
    """

    def __init__(self, n_nodes, edge_src, edge_dst, edge_w, passage_vid, fact_subj_vid, fact_obj_vid,
                 ent_chunk_count, fact_emb, passage_emb, device: int = 0, damping: float = 0.5,
                 linking_top_k: int = 5, passage_node_weight: float = 0.05, retrieval_top_k: int = 200,
                 engine: Optional[Engine] = None):
        self.engine = engine or Engine(device)
        self.engine.load_graph(n_nodes, edge_src, edge_dst, edge_w)
        self.engine.load_tables(passage_vid, fact_subj_vid, fact_obj_vid, ent_chunk_count)
        self.engine.load_embeddings(fact_emb, passage_emb)
        self.damping = damping
        self.linking_top_k = linking_top_k
        self.passage_node_weight = passage_node_weight
        self.retrieval_top_k = retrieval_top_k

    def retrieve(self, q_fact, q_pass, fact_filter: Optional[FactFilter] = None, topk: Optional[int] = None):
        k = self.linking_top_k
        topk = min(topk or self.retrieval_top_k, 2048)
        idx, score, nv = self.engine.stage_a(q_fact, k)
        if fact_filter is not None:
            for q in range(idx.shape[0]):
                keep = list(fact_filter(q, idx[q, :nv[q]].tolist(), score[q, :nv[q]].tolist()))
                kept_i = [idx[q, j] for j in keep]
                kept_s = [score[q, j] for j in keep]
                idx[q] = -1
                idx[q, :len(kept_i)] = kept_i
                score[q, :len(kept_s)] = kept_s
        ids, scores = self.engine.stage_b(q_pass, idx, score, None, self.damping, self.passage_node_weight,
                                          self.linking_top_k, topk)
        return ids, scores, idx, score
