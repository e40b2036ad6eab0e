#!/usr/bin/env python
"""Benchmark of the HippoRAG retrieval hot path on B200 (contract: see the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C1|C2|C3|C5] [--impl reference]
                    [--dump-outputs DIR]

A *step* = one batch of ``--queries`` queries through the whole path
(stage A: query x fact similarity + top-5 -> identity recognition-memory filter -> stage B:
query x passage similarity + seeds + PPR + top-200) on the workload's knowledge graph.
``value`` = queries/s with inputs resident in HBM (device pointers); ``e2e`` = the same through
the host-buffer C-ABI calls (pinned host queries in, top-k ids/scores out, copies timed).
Timing: CUDA events recorded on the library's own launch stream, barrier + synchronize on both
sides, max over ranks.  Inputs (hundreds of MB of state + GBs of embeddings) exceed L2, so no
explicit L2 flush is needed between iterations (C1 is the exception and says so).

Workloads (BASELINE.json configs): C1 = MuSiQue-1k (the reference's own index() output, committed as
tests/golden/musique1k.npz; 64 queries), C2 / C3 = synthetic uniform KGs, C5 = 10M-node power-law KG with
1024-d embeddings (facts uploaded streamed, bf16 planes only).

N > 1 (launched under torch.distributed.run): ``value`` = *replicas* -- every rank holds the whole graph and
its own batch of queries (queries are independent units, SURVEY.md 8(e)); no data-path collective;
``scaling: weak``.  The same line then carries a ``sharded`` object: BASELINE config #4, the SAME graph
node-range-sharded over the N GPUs (rows of P and rows of the fact matrix split by range, all ranks
working on one batch; fused peer-store exchange per sweep, K5).  ``--shard node`` makes the sharded run the
headline instead.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "C1": dict(golden=True, dim=768, queries=64, topology="real",
               desc="MuSiQue-1k: the reference index() graph (11,325 nodes / 33,269 edges / 10,734 facts / 1,000 "
                    "passages), 768-d seeded mock embeddings, 64 queries"),
    "C2": dict(n_nodes=100_000, n_edges=1_000_000, dim=768, queries=1_000, topology="uniform",
               desc="synthetic 100k-node / 1M-edge KG, 768-d embeddings, 1k queries"),
    "C3": dict(n_nodes=1_000_000, n_edges=10_000_000, dim=768, queries=10_000, topology="uniform",
               desc="synthetic 1M-node / 10M-edge KG, 768-d embeddings, 10k batched queries"),
    "C5": dict(n_nodes=10_000_000, n_edges=100_000_000, dim=1024, queries=128, topology="powerlaw", streamed=True,
               desc="synthetic 10M-node / 100M-edge power-law KG, 1024-d embeddings"),
}
TOPK, LINK_TOP_K, DAMPING, PNW = 200, 5, 0.5, 0.05
DTYPE = "bf16x4-split tcgen05 GEMM (fp32 accumulate) + fp16-state PPR with fp32 residual refinement; fp32 outputs"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def emb_chunk_torch(rows_lo, rows_hi, dim, seed, device):
    """Rows [rows_lo, rows_hi) of a seeded unit-Gaussian matrix; one generator per 2^18-row block so any
    block can be regenerated on its own (streamed / sharded uploads)."""
    import torch
    step = 1 << 18
    assert rows_lo % step == 0
    out = torch.empty((rows_hi - rows_lo, dim), dtype=torch.float32, device=device)
    for lo in range(rows_lo, rows_hi, step):
        hi = min(rows_hi, lo + step)
        g = torch.Generator(device=device)
        g.manual_seed(seed * 100_003 + lo // step)
        x = torch.randn((hi - lo, dim), generator=g, device=device, dtype=torch.float32)
        out[lo - rows_lo:hi - rows_lo] = x / x.norm(dim=1, keepdim=True)
    return out


def gen_embeddings_torch(rows, dim, seed, device):
    return emb_chunk_torch(0, rows, dim, seed, device)


def perturb_torch(base, g, device):
    import torch
    z = torch.randn(base.shape, generator=g, device=device, dtype=torch.float32)
    z = z / z.norm(dim=1, keepdim=True)
    q = base + 0.5 * z
    return (q / q.norm(dim=1, keepdim=True)).contiguous()


class Workload:
    """Graph + tables + embeddings (or an embedding chunk generator) + queries of one config."""
    pass


def build_workload(name, n_queries, device, rank, want_embeddings=True):
    import torch
    from hipporag_b200 import synth
    from hipporag_b200.engine import build_transition_csr
    w = WORKLOADS[name]
    wl = Workload()
    wl.name, wl.cfg = name, w
    t0 = time.time()
    if w.get("golden"):
        g = dict(np.load(os.path.join(ROOT, "tests", "golden", "musique1k.npz")))
        n = int(g["n_nodes"])
        kg = synth.SynthKG(n, n - len(g["passage_vid"]), len(g["passage_vid"]), g["edge_src"], g["edge_dst"], g["edge_w"],
                           g["passage_vid"], g["fact_subj_vid"], g["fact_obj_vid"], g["ent_chunk_count"],
                           np.zeros(len(g["fact_subj_vid"]), np.int32))
        wl.kg = kg
        wl.csr = build_transition_csr(n, kg.edge_src, kg.edge_dst, kg.edge_w)
        dim = int(g["dim"])
        wl.fe = torch.from_numpy(synth.seeded_unit_vectors(g["fact_seed"], dim)).to(device)
        wl.pe = torch.from_numpy(synth.seeded_unit_vectors(g["passage_seed"], dim)).to(device)
        reps = -(-n_queries // len(g["qfact_seed"]))
        qf = np.tile(synth.seeded_unit_vectors(g["qfact_seed"], dim), (reps, 1))[:n_queries]
        qp = np.tile(synth.seeded_unit_vectors(g["qpass_seed"], dim), (reps, 1))[:n_queries]
        wl.qf, wl.qp = torch.from_numpy(qf).to(device), torch.from_numpy(qp).to(device)
        wl.fact_chunks = None
        log(f"[bench r{rank}] graph C1 (tests/golden/musique1k.npz): N={n} E={kg.n_edges} F={kg.n_facts} P={kg.n_pass}")
        return wl
    kg = synth.make_kg(w["n_nodes"], w["n_edges"], seed=0, topology=w["topology"])
    wl.kg = kg
    wl.csr = build_transition_csr(kg.n_nodes, kg.edge_src, kg.edge_dst, kg.edge_w)
    deg = np.diff(wl.csr[0])
    log(f"[bench r{rank}] graph {name}: N={kg.n_nodes} E={kg.n_edges} nnz={wl.csr[1].shape[0]} F={kg.n_facts} "
        f"P={kg.n_pass} max degree {int(deg.max())} ({time.time() - t0:.1f}s)")
    dim = w["dim"]
    g = torch.Generator(device=device)
    g.manual_seed(1000 + rank)
    j = torch.randint(0, kg.n_facts, (n_queries,), generator=g, device=device)
    i = torch.from_numpy(kg.fact_passage).to(device)[j].long()
    wl.pe = gen_embeddings_torch(kg.n_pass, dim, 101, device) if want_embeddings else None
    if w.get("streamed"):
        # facts never exist as one fp32 matrix: blocks are generated, handed to the engine, and dropped; the rows the
        # queries are planted on are picked up on the way
        wl.fe = None
        step = 1 << 18
        base_f = torch.empty((n_queries, dim), dtype=torch.float32, device=device)
        jl = j.cpu().numpy()

        def fact_chunks(lo_hi=None):
            lo0, hi0 = lo_hi if lo_hi else (0, kg.n_facts)
            for lo in range((lo0 // step) * step, hi0, step):
                hi = min(kg.n_facts, lo + step)
                blk = emb_chunk_torch(lo, hi, dim, 100, device)
                yield lo, blk
        wl.fact_chunks = fact_chunks
        # query bases: regenerate only the blocks that hold a planted fact
        for lo in sorted(set(((jl // step) * step).tolist())):
            hi = min(kg.n_facts, lo + step)
            blk = emb_chunk_torch(lo, hi, dim, 100, device)
            sel = np.nonzero((jl >= lo) & (jl < hi))[0]
            base_f[torch.from_numpy(sel).to(device)] = blk[torch.from_numpy(jl[sel] - lo).to(device)]
            del blk
        wl.qf = perturb_torch(base_f, g, device)
    else:
        wl.fe = gen_embeddings_torch(kg.n_facts, dim, 100, device) if want_embeddings else None
        wl.fact_chunks = None
        wl.qf = perturb_torch(wl.fe[j], g, device) if want_embeddings else None
    if want_embeddings:
        wl.qp = perturb_torch(wl.pe[i], g, device)
    return wl


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except Exception:
                continue
            for k, nm in enumerate(names):
                if len(r) > 5 + k and r[5 + k].strip().lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


def ppr_bytes_per_sweep(n_rows, nnz, B):
    """SURVEY.md 8(d): nnz*(4 col + 4 val) + (N+1)*4 row_ptr + B*N*4*3 (read X, write Y, read V)."""
    return nnz * 8 + (n_rows + 1) * 4 + 3 * n_rows * B * 4


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is entitled to every host core."""
    n = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=n)
    except Exception:
        pass
    try:
        import torch
        torch.set_num_threads(n)
    except Exception:
        pass
    return n


def _cpu_inputs(wl):
    import scipy.sparse as sp
    from oracle import retrieve
    kg = wl.kg
    row_ptr, col, val = wl.csr
    P = sp.csr_matrix((val.astype(np.float64), col, row_ptr), shape=(kg.n_nodes, kg.n_nodes))
    tb = retrieve.Tables(kg.n_nodes, kg.passage_vid, kg.fact_subj_vid, kg.fact_obj_vid, kg.ent_chunk_count)
    return P, tb


def cpu_baseline_leg(wl, fe_host, pe_host, qf_host, qp_host, n_sample):
    """The reference's per-query CPU path (oracle/cpu_reference.py: serial loop, fp32 sgemv, f64 PPR to 1e-10)."""
    use_all_host_threads()
    from oracle import cpu_reference
    P, tb = _cpu_inputs(wl)
    ids, scores, secs, parts = cpu_reference.retrieve_serial(P, tb, fe_host, pe_host, qf_host[:n_sample],
                                                             qp_host[:n_sample], LINK_TOP_K, PNW, DAMPING, TOPK)
    return n_sample / secs, secs, parts, ids, scores


def cpu_best_effort_leg(wl, fe_host, pe_host, qf_host, qp_host, n_sample):
    """SURVEY.md 8(d)(2): the best a careful numpy/scipy rewrite does on the host cores -- batched sgemm, fp32 CSR
    SpMM Chebyshev PPR over all cores, argpartition -- so the GPU ratio is not quoted against a strawman only."""
    cores = use_all_host_threads()
    from oracle import cpu_reference
    P, tb = _cpu_inputs(wl)
    ids, scores, secs, parts, info = cpu_reference.retrieve_vectorized(
        P, tb, fe_host, pe_host, qf_host[:n_sample], qp_host[:n_sample], LINK_TOP_K, PNW, DAMPING, TOPK,
        batch=min(64, n_sample), threads=cores)
    return n_sample / secs, secs, parts, info, ids


def run_reference_arm(args, rank, world):
    """`--impl reference`: the reference's CPU implementation of the path on the host cores."""
    if rank != 0:
        return
    import torch
    use_all_host_threads()
    w = WORKLOADS[args.workload]
    n_sample = args.ref_queries
    wl = build_workload(args.workload, n_sample * (args.steps + args.warmup), "cpu", 0)
    fe, pe, qf, qp = wl.fe.numpy(), wl.pe.numpy(), wl.qf.numpy(), wl.qp.numpy()
    times = []
    for s in range(args.warmup + args.steps):
        lo = s * n_sample
        qps, secs, parts, _, _ = cpu_baseline_leg(wl, fe, pe, qf[lo:lo + n_sample], qp[lo:lo + n_sample], n_sample)
        log(f"[reference] step {s}: {n_sample} queries in {secs:.2f}s ({parts})")
        if s >= args.warmup:
            times.append(secs)
    total = sum(times)
    value = n_sample * args.steps / total
    cores = os.cpu_count() or 1
    line = {
        "impl": "reference", "metric": "retrieval queries/sec (batched PPR+embed-sim)", "value": value,
        "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 similarity + f64 PPR (the reference's own dtypes)", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {w['desc']}", "queries_per_step": n_sample, "topk": TOPK,
                   "linking_top_k": LINK_TOP_K, "damping": DAMPING, "filter": "identity"},
        "cpu_baseline": {"value": value, "unit": "queries/s", "cores": cores, "kind": "port",
                         "sample": f"{n_sample} queries per step, serial per-query loop as HippoRAG.retrieve; "
                                   f"fp32 BLAS sgemv (threads={torch.get_num_threads()}) + scipy f64 PPR to 1e-10 "
                                   "(python-igraph/PRPACK not installable offline)"},
        "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def load_engine(eng, wl, args_obj=None):
    kg = wl.kg
    row_ptr, col, val = wl.csr
    eng.load_graph_csr(kg.n_nodes, row_ptr, col, val)
    eng.load_tables(kg.passage_vid, kg.fact_subj_vid, kg.fact_obj_vid, kg.ent_chunk_count)
    if wl.fact_chunks is not None:
        lo_hi = None
        if eng.world > 1:
            chunk = -(-kg.n_facts // eng.world)
            lo_hi = (min(kg.n_facts, eng.rank * chunk), min(kg.n_facts, (eng.rank + 1) * chunk))
        eng.load_embeddings_streamed(0, kg.n_facts, wl.cfg["dim"], wl.fact_chunks(lo_hi))
        eng.load_embeddings_streamed(1, kg.n_pass, wl.cfg["dim"], [(0, wl.pe)])
    else:
        eng.load_embeddings(wl.fe, wl.pe)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, ids, scores):
    """What ``retrieve_resident`` hands its caller: top-k passage ids (as float64, exact for int32) and scores
    (float32), one row per query.  Batches too large for DUMP_BYTES keep a fixed seeded sample of rows, listed in
    ``rows.npy``, so two builds run with the same arguments can be compared row for row."""
    row_bytes = ids.shape[1] * 8 + scores.shape[1] * 4 + 8
    rows = np.arange(ids.shape[0])
    if rows.size * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(rows.size, DUMP_BYTES // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "topk_ids.npy"), ids[rows].astype(np.float64))
    np.save(os.path.join(out_dir, "topk_scores.npy"), scores[rows].astype(np.float32))
    log(f"[bench] outputs of the last timed step ({rows.size} of {ids.shape[0]} queries) written to {out_dir}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C3", choices=sorted(WORKLOADS))
    ap.add_argument("--queries", type=int, default=0, help="queries per step (default: the workload's)")
    ap.add_argument("--shard", default="replicas", choices=["replicas", "node"])
    ap.add_argument("--no-sharded-leg", action="store_true", help="N > 1: skip the node-range-sharded measurement")
    ap.add_argument("--no-p2p", action="store_true", help="node sharding: NCCL all-gather per sweep instead of fused peer stores")
    ap.add_argument("--ppr-batch", type=int, default=0)
    ap.add_argument("--ppr-iters", type=int, default=0)
    ap.add_argument("--ppr-method", default="", choices=["", "power", "chebyshev"])
    ap.add_argument("--ppr-precision", default="", choices=["", "fp32", "mixed"])
    ap.add_argument("--cpu-sample", type=int, default=8, help="queries in the cpu_baseline sample (0 = skip)")
    ap.add_argument("--cpu-best-effort-sample", type=int, default=128, help="queries in the best-effort CPU leg (0 = skip)")
    ap.add_argument("--ref-queries", type=int, default=4, help="queries per step of --impl reference")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the top-k ids and scores of the last timed step to DIR/*.npy (rank 0's batch)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    # one JSON line on stdout: NCCL prints its version banner (levels VERSION and WARN) and its INFO log there
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
        del os.environ["NCCL_DEBUG"]
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from hipporag_b200 import Engine, PPR_CHEBYSHEV, PPR_FP32, PPR_MIXED, PPR_POWER

    w = WORKLOADS[args.workload]
    Q = args.queries or w["queries"]
    nnz = None
    side = dist.new_group(backend="gloo") if world > 1 else None   # host-side object exchange (IPC handles)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def make_engine(mode, wl):
        eng = Engine(local_rank, shard_mode=1 if mode == "node" else 0)
        if world > 1 and mode == "node":
            ids = [Engine.new_comm_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            eng.init_comm(ids[0], rank, world)
        kg = wl.kg
        row_ptr, col, val = wl.csr
        eng.load_graph_csr(kg.n_nodes, row_ptr, col, val)
        if world > 1 and mode == "node" and not args.no_p2p:
            handles = [None] * world
            dist.all_gather_object(handles, eng.p2p_export(), group=side)
            eng.p2p_import(handles)
        eng.load_tables(kg.passage_vid, kg.fact_subj_vid, kg.fact_obj_vid, kg.ent_chunk_count)
        if wl.fact_chunks is not None:
            lo_hi = None
            if eng.world > 1:
                chunk = -(-kg.n_facts // eng.world)
                lo_hi = (min(kg.n_facts, eng.rank * chunk), min(kg.n_facts, (eng.rank + 1) * chunk))
            eng.load_embeddings_streamed(0, kg.n_facts, w["dim"], wl.fact_chunks(lo_hi))
            eng.load_embeddings_streamed(1, kg.n_pass, w["dim"], [(0, wl.pe)])
        else:
            eng.load_embeddings(wl.fe, wl.pe)
        eng.set_options(ppr_method={"": None, "power": PPR_POWER, "chebyshev": PPR_CHEBYSHEV}[args.ppr_method],
                        ppr_iters=args.ppr_iters or None, ppr_batch=args.ppr_batch or None,
                        ppr_precision={"": None, "fp32": PPR_FP32, "mixed": PPR_MIXED}[args.ppr_precision])
        return eng

    def measure(mode, wl):
        """-> dict(ms_total, st, clocks, e2e, out_ids) for one parallelism mode on workload wl."""
        eng = make_engine(mode, wl)
        out_ids = torch.empty((Q, TOPK), dtype=torch.int32, device=device)
        out_scores = torch.empty((Q, TOPK), dtype=torch.float32, device=device)
        lib_stream = torch.cuda.ExternalStream(eng.stream_ptr, device=device)

        def resident_step():
            eng.retrieve_resident(wl.qf, wl.qp, out_ids, out_scores, DAMPING, PNW, LINK_TOP_K, TOPK)

        h_qf, h_qp = wl.qf.cpu().pin_memory(), wl.qp.cpu().pin_memory()
        h_qf_np, h_qp_np = h_qf.numpy(), h_qp.numpy()

        def e2e_step():
            idx, score, nv = eng.stage_a(h_qf_np, LINK_TOP_K)           # H2D queries, D2H top facts
            # identity recognition-memory filter on the host (rerank.py:108 stand-in)
            return eng.stage_b(h_qp_np, idx, score, None, DAMPING, PNW, LINK_TOP_K, TOPK)   # D2H top-k

        def timed(fn, steps):
            barrier()
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(lib_stream)
            for _ in range(steps):
                fn()
            e1.record(lib_stream)
            barrier()
            ms = e0.elapsed_time(e1)
            if world > 1:
                t = torch.tensor([ms], device=device, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            return ms

        for _ in range(args.warmup):
            resident_step()
        eng.reset_stats()
        sampler = ClockSampler(local_rank) if rank == 0 else None
        ms_total = timed(resident_step, args.steps)
        clocks = sampler.stop() if sampler else None
        st = eng.stats()
        e2e = None
        if not args.no_e2e:
            for _ in range(min(args.warmup, 1) or 1):
                e2e_step()
            eng.reset_stats()
            ms_e2e = timed(e2e_step, args.steps)
            st2 = eng.stats()
            n_eff = world if mode == "replicas" else 1
            e2e = {"value": Q * args.steps * n_eff / (ms_e2e / 1000.0), "unit": "queries/s",
                   "h2d_bytes_per_step": int(st2["h2d_bytes"] // args.steps),
                   "d2h_bytes_per_step": int(st2["d2h_bytes"] // args.steps), "ms_per_step": ms_e2e / args.steps}
        res = dict(ms_total=ms_total, st=st, clocks=clocks, e2e=e2e, out_ids=out_ids[:max(args.cpu_sample, 8)].cpu().numpy(),
                   h_qf=h_qf_np, h_qp=h_qp_np)
        if args.dump_outputs and mode == head_mode:
            res["dump"] = (out_ids.cpu().numpy(), out_scores.cpu().numpy())   # still the last timed step's results
        eng.close()
        del eng
        torch.cuda.empty_cache()
        return res

    head_mode = args.shard if world > 1 else "replicas"
    # replicas: every rank has its own queries; node sharding: all ranks cooperate on the SAME batch
    wl = build_workload(args.workload, Q, device, rank if head_mode == "replicas" else 0)
    nnz = int(wl.csr[1].shape[0])
    kg = wl.kg
    main_res = measure(head_mode, wl)
    sharded_res = None
    if world > 1 and head_mode == "replicas" and not args.no_sharded_leg:
        del wl
        torch.cuda.empty_cache()
        wl = build_workload(args.workload, Q, device, 0)      # the same batch on every rank
        sharded_res = measure("node", wl)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peaks()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *main_res["dump"])

    def roofline_of(res, mode):
        st = res["st"]
        sweeps = max(int(st["ppr_sweeps"]), 1)
        Bavg = st["ppr_columns"] / sweeps
        sharded = world > 1 and mode == "node"
        n_rows_local = -(-kg.n_nodes // world) if sharded else kg.n_nodes
        nnz_local = nnz // world if sharded else nnz
        bytes_sweep = ppr_bytes_per_sweep(n_rows_local, nnz_local, Bavg)
        ms_sweep = st["ms_ppr"] / sweeps
        achieved = bytes_sweep / (ms_sweep * 1e-3) / 1e9
        mixed = abs(Bavg - 32.0) < 1e-6
        bytes_layout = (nnz_local * 8 + (n_rows_local + 1) * 4 + 3 * n_rows_local * Bavg * 2) if mixed else bytes_sweep
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "k1_traffic.json")
        if os.path.exists(tpath) and not sharded:
            try:
                tj = json.load(open(tpath))
                traffic = tj.get(f"{args.workload}_B{int(Bavg)}")
                traffic_src = tj.get("source")
            except Exception:
                traffic = None
        return {"kernel": ("k_sweep_h (K1m: CSR SpMM PPR sweep, fp16 state / fp32 math, B=32)" if mixed else
                           "k_sweep_rows (K1: CSR SpMM PPR sweep, fp32 state)"),
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "bytes_per_launch": bytes_sweep, "bytes_per_launch_in_this_layout": bytes_layout,
                "achieved_in_this_layout": bytes_layout / (ms_sweep * 1e-3) / 1e9,
                "ms_per_launch": ms_sweep, "launches": sweeps, "batch_width": Bavg,
                "note": "achieved = SURVEY 8(d) algorithmic bytes (fp32 vectors: nnz*8 + (N+1)*4 + 3*N*B*4) / in-step "
                        "average sweep time (ms_ppr / sweeps: every kernel between the first and the last sweep of a "
                        "solve is inside it)"}

    def stage_ms(res):
        return {k: round(res["st"][k] / args.steps, 3) for k in ("ms_sim_fact", "ms_select_fact", "ms_sim_passage",
                                                                  "ms_seed", "ms_ppr", "ms_topk", "ms_comm")}

    st = main_res["st"]
    n_eff = world if head_mode == "replicas" else 1
    value = Q * args.steps * n_eff / (main_res["ms_total"] / 1000.0)
    roof = roofline_of(main_res, head_mode)
    mixed = abs(roof["batch_width"] - 32.0) < 1e-6
    line = {
        "metric": "retrieval queries/sec (batched PPR+embed-sim)", "value": value, "unit": "queries/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": main_res["ms_total"] / args.steps,
        "higher_is_better": True, "scaling": "weak" if head_mode == "replicas" else "strong",
        "vs_baseline": None, "dtype": DTYPE, "data": "synthetic" if not w.get("golden") else
        "the reference's own index() graph of MuSiQue-1k (committed fixture) + seeded mock embeddings",
        "config": {"workload": f"{args.workload}: {w['desc']}", "queries_per_step_per_gpu": Q, "topk": TOPK,
                   "linking_top_k": LINK_TOP_K, "damping": DAMPING, "passage_node_weight": PNW,
                   "filter": "identity", "parallelism": f"{head_mode}x{world}" + (
                       "" if head_mode == "replicas" or world == 1 else
                       (" (NCCL all-gather per sweep)" if args.no_p2p else " (fused peer-store exchange)")),
                   "ppr": {"method": "chebyshev" if args.ppr_method in ("", "chebyshev") else "power",
                           "precision": "fp16 state + fp32 refinement (sweeps derived from damping: 8+1+7)" if mixed else "fp32",
                           "sweeps_per_query": st["ppr_columns"] / max(Q * args.steps, 1), "batch_width": roof["batch_width"],
                           "residual_check": {"measured_rel_l1_residual_of_fp16_solve": st.get("ppr_residual"),
                                              "a_posteriori_error_bound": st.get("ppr_error_bound")}},
                   "l2": ("inputs larger than L2 (no flush needed)" if not w.get("golden") else
                          "C1 fits L2 entirely: numbers are L2-resident by nature of the config"),
                   "stage_ms_per_step": stage_ms(main_res)},
        "clocks": main_res["clocks"], "e2e": main_res["e2e"], "gpu_launches": int(st["kernel_launches"]),
        "roofline": roof,
    }
    if sharded_res is not None:
        sv = Q * args.steps / (sharded_res["ms_total"] / 1000.0)
        sroof = roofline_of(sharded_res, "node")
        line["sharded"] = {
            "config": f"BASELINE config #4: {args.workload} graph node-range-sharded over {world} GPUs (rows of P and rows of "
                      "the fact matrix by range; every rank works on the same batch)",
            "value": sv, "unit": "queries/s", "scaling": "strong", "ms_per_step": sharded_res["ms_total"] / args.steps,
            "exchange": "NCCL all-gather per sweep" if args.no_p2p else
                        "K5: sweep epilogue stores rows into every peer over NVLink; epoch flags inside the sweep kernel",
            "stage_ms_per_step": stage_ms(sharded_res), "ms_comm_per_step": stage_ms(sharded_res)["ms_comm"],
            "speedup_vs_one_replica": sv / (value / world), "roofline_per_gpu": sroof,
            "e2e": sharded_res["e2e"], "clocks": sharded_res["clocks"],
            "nvlink_bytes_in_per_gpu_per_sweep": int((world - 1) * -(-kg.n_nodes // world) * 64),
        }
    if world == 1 and args.cpu_sample > 0 and wl.fe is not None:
        fe_h, pe_h = wl.fe.cpu().numpy(), wl.pe.cpu().numpy()
        ns = min(args.cpu_sample, Q)
        qps, secs, parts, cids, cscores = cpu_baseline_leg(wl, fe_h, pe_h, main_res["h_qf"], main_res["h_qp"], ns)
        gpu_ids = main_res["out_ids"]
        agree = float(np.mean([len(set(gpu_ids[i].tolist()) & set(cids[i].tolist())) / min(TOPK, kg.n_pass)
                               for i in range(ns)]))
        line["cpu_baseline"] = {"value": qps, "unit": "queries/s", "cores": os.cpu_count() or 1, "kind": "port",
                                "sample": f"first {ns} queries of the step, serial per-query loop as HippoRAG.retrieve "
                                          f"(fp32 BLAS sgemv, scipy f64 PPR to 1e-10); {secs:.1f}s; stages {parts}",
                                "topk_overlap_with_gpu": agree}
        nb = min(args.cpu_best_effort_sample, Q)
        if nb > 0:
            bq, bsecs, bparts, binfo, bids = cpu_best_effort_leg(wl, fe_h, pe_h, main_res["h_qf"], main_res["h_qp"], nb)
            line["cpu_baseline"]["best_effort"] = {
                "value": bq, "unit": "queries/s", "cores": binfo["threads"], "kind": "port (vectorised rewrite, NOT how "
                "the reference runs)", "sample": f"first {nb} queries, batches of {binfo['batch']}: sgemm + argpartition, "
                f"fp32 CSR SpMM Chebyshev PPR ({binfo['sweeps']} sweeps, {binfo['spmm']}); {bsecs:.1f}s; stages {bparts}",
                "gpu_over_best_effort_cpu": value / bq}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
