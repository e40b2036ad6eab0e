"""CPU-only tests of host-side product code: the synthetic KG generator, the drop-in's table
extraction (against the harness run of the reference), bench.py's bookkeeping and reference arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_synthetic_kg_matches_the_documented_shape():
    from hipporag_b200 import synth
    kg = synth.make_kg(20_000, 200_000, seed=1)
    assert kg.n_pass == 2_000 and kg.n_ent == 18_000
    assert abs(kg.n_edges - 200_000) < 2_000
    # ~55 % of the edges are fact edges emitted as parallel pairs (s,o)/(o,s) with equal integer weights
    F = kg.n_facts
    assert abs(2 * F / kg.n_edges - 0.55) < 0.01
    assert np.array_equal(kg.edge_src[:F], kg.edge_dst[F:2 * F]) and np.array_equal(kg.edge_dst[:F], kg.edge_src[F:2 * F])
    assert np.array_equal(kg.edge_w[:F], kg.edge_w[F:2 * F]) and np.all(kg.edge_w[:F] == np.round(kg.edge_w[:F]))
    # vertex order: entities then passages; passage edges have weight 1; synonymy weights in [0.8, 1)
    assert np.array_equal(kg.passage_vid, np.arange(kg.n_ent, kg.n_nodes))
    pe = slice(2 * F, 2 * F + int(round(0.35 * 200_000)))
    assert np.all(kg.edge_src[pe] >= kg.n_ent) and np.all(kg.edge_dst[pe] < kg.n_ent) and np.all(kg.edge_w[pe] == 1.0)
    syn = kg.edge_w[pe.stop:]
    assert syn.size > 0 and syn.min() >= 0.8 and syn.max() < 1.0
    # ent_chunk_count = passage degree; 0.1 % of the entities are isolated (sinks)
    deg = np.zeros(kg.n_nodes, dtype=np.int64)
    np.add.at(deg, kg.edge_src, 1)
    np.add.at(deg, kg.edge_dst, 1)
    assert np.all(deg[kg.n_ent - 18:kg.n_ent] == 0)
    cnt = np.zeros(kg.n_nodes, dtype=np.int64)
    np.add.at(cnt, kg.edge_dst[pe], 1)
    assert np.array_equal(cnt, kg.ent_chunk_count)
    # determinism
    kg2 = synth.make_kg(20_000, 200_000, seed=1)
    assert np.array_equal(kg.edge_src, kg2.edge_src) and np.array_equal(kg.edge_w, kg2.edge_w)
    # planted queries are unit vectors close to their fact / passage
    fe, pe_ = synth.unit_rows(kg.n_facts, 32, 3), synth.unit_rows(kg.n_pass, 32, 4)
    qf, qp, j = synth.make_queries(kg, fe, pe_, 50, seed=5)
    np.testing.assert_allclose(np.linalg.norm(qf, axis=1), 1.0, atol=1e-5)
    assert np.all(np.einsum("ij,ij->i", qf, fe[j]) > 0.8)
    pl = synth.make_kg(5_000, 50_000, seed=2, topology="powerlaw")
    d = np.bincount(np.concatenate([pl.edge_src, pl.edge_dst]), minlength=pl.n_nodes)
    assert d.max() > 20 * np.median(d[d > 0])            # a heavy tail


def test_roofline_byte_model():
    sys.path.insert(0, ROOT)
    import bench
    # SURVEY.md 8(d): nnz*8 + (N+1)*4 + 3*N*B*4
    assert bench.ppr_bytes_per_sweep(1_000_000, 14_499_972, 16) == 14_499_972 * 8 + 1_000_001 * 4 + 3 * 1_000_000 * 16 * 4
    peak, src = bench.measured_peaks()
    assert 3000 < peak < 9000 and ("measured" in src or "fallback" in src)


def test_dropin_table_extraction_matches_the_harness(tmp_path):
    """accelerate.extract_tables (product) and oracle.ref_harness.extract_tables (test infrastructure) are
    written independently from the same reference lines; on the reference's own object (replayed from
    tests/golden/reference_rag150.npz, which holds what the harness extracted from it) they must agree."""
    from tests import fake_hipporag
    fake_hipporag.install_stub_package()
    from hipporag_b200.accelerate import extract_tables
    g, rag = fake_hipporag.load_recorded_rag(str(tmp_path))
    rag.prepare_retrieval_objects()
    want = {k: g[k] for k in ("edge_src", "edge_dst", "edge_w")}
    want.update({k: g["harness_" + k] for k in ("n_nodes", "passage_vid", "fact_subj_vid", "fact_obj_vid",
                                                "ent_chunk_count")})
    got = extract_tables(rag)
    for k in ("n_nodes", "edge_src", "edge_dst", "edge_w", "passage_vid", "fact_subj_vid", "fact_obj_vid",
              "ent_chunk_count"):
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), k
    assert [str(f) for f in got["facts"]] == g["fact_texts"].tolist()
    assert (got["fact_subj_vid"] >= 0).all() and (got["ent_chunk_count"][got["passage_vid"]] == 0).all()


def test_bench_dump_outputs_fixed_sample_within_budget(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(1)
    ids = rng.integers(0, 1 << 30, (300, 200)).astype(np.int32)
    scores = rng.random((300, 200)).astype(np.float32)
    bench.dump_outputs(str(tmp_path / "all"), ids, scores)
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "topk_ids.npy"), ids)
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "topk_scores.npy"), scores)
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * (200 * 12 + 8))      # room for 100 of the 300 rows
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), ids, scores)
    rows = np.load(tmp_path / "a" / "rows.npy").astype(np.int64)
    assert rows.size == 100 and np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))
    got = np.load(tmp_path / "a" / "topk_ids.npy")
    assert got.dtype == np.float64 and np.array_equal(got, ids[rows])
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES + 3 * 128


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "C2",
                          "--steps", "1", "--warmup", "0", "--ref-queries", "2"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_sweep_counts_are_derived_from_damping_and_tolerance():
    """config_utils.py:192 makes damping configurable and PRPACK converges whatever it is; the library derives its
    sweep counts from (damping, tol) -- hrag_plan_sweeps is that rule as a pure host function (no GPU needed)."""
    import math
    from hipporag_b200.engine import plan_sweeps
    p = plan_sweeps(0.5)                                     # the reference default: 8 + 1 + 7 fp16 sweeps, or 14 fp32
    assert p["solver"] == "mixed" and p["mixed_sweeps"] == (8, 1, 7) and p["fp32_sweeps"] == 14
    assert p["predicted_error"] < 1e-6
    assert plan_sweeps(0.5, batch=8)["solver"] == "fp32"      # <= 16 columns: the fp32 solver at its own width
    # the Chebyshev rate sigma = a / (1 + sqrt(1 - a^2)): fp32 sweeps = ceil(log(1e-8) / log(sigma))
    for a in (0.2, 0.5, 0.7, 0.85, 0.95):
        sigma = a / (1 + math.sqrt(1 - a * a))
        assert plan_sweeps(a)["fp32_sweeps"] == math.ceil(math.log(1e-8) / math.log(sigma) - 1e-9)
    # damping 0.85: one refinement round cannot reach 1e-6 -> the fp32 solver, 32 sweeps (14 would leave ~3e-4)
    p85 = plan_sweeps(0.85)
    assert p85["solver"] == "fp32" and p85["fp32_sweeps"] == 32
    assert plan_sweeps(0.85, tol=1e-5)["solver"] == "mixed"   # a looser tolerance lets the fp16 solver back in
    # monotone in the damping and in the tolerance
    sweeps = [plan_sweeps(a)["fp32_sweeps"] for a in (0.3, 0.5, 0.7, 0.9)]
    assert sweeps == sorted(sweeps) and len(set(sweeps)) == 4
    assert plan_sweeps(0.5, tol=1e-4)["fp32_sweeps"] < plan_sweeps(0.5, tol=1e-8)["fp32_sweeps"]
    # iters > 0 pins the counts (mixed: m1 = iters, m2 = iters - 1)
    pin = plan_sweeps(0.5, iters=10)
    assert pin["fp32_sweeps"] == 10 and pin["mixed_sweeps"] == (10, 1, 9)
    from hipporag_b200 import HragError
    with pytest.raises(HragError):
        plan_sweeps(1.0)


def test_index_cache_roundtrip_and_invalidation(tmp_path):
    """hipporag_b200/cache.py (SURVEY.md 8(f)-3) on a duck-typed rag (no reference checkout needed): the CSR + tables +
    fact triples written beside graph.pickle are reused while the index fingerprint is unchanged and rebuilt when the
    graph, the fact list or the passage list changes."""
    import sys
    from tests import fake_hipporag
    fake_hipporag.install_stub_package()
    import hipporag_b200
    from hipporag_b200 import cache, synth
    from hipporag_b200.engine import build_transition_csr

    class RecordingEngine:                       # Engine's upload interface, nothing else
        dim = 8

        def __init__(self):
            self.calls = []

        def load_graph_csr(self, n, row_ptr, col, val):
            self.calls.append(("csr", n, np.asarray(row_ptr).copy(), np.asarray(col).copy(), np.asarray(val).copy()))

        def load_tables(self, pv, fs, fo, cc):
            self.calls.append(("tables", np.asarray(pv).copy(), np.asarray(fs).copy(), np.asarray(fo).copy(), np.asarray(cc).copy()))

        def load_embeddings(self, fe, pe):
            self.calls.append(("emb", fe.shape, pe.shape))

        def set_options(self, **kw):
            pass

    kg = synth.make_kg(400, 4000, seed=3)
    fe, pe = synth.unit_rows(kg.n_facts, 8, 1), synth.unit_rows(kg.n_pass, 8, 2)
    rag = fake_hipporag.FakeRag(kg, fe, pe, fe[:1], pe[:1], ["q"])
    rag.working_dir = str(tmp_path)
    acc_mod = sys.modules["hipporag_b200.accelerate"]
    n_extract = []
    real_extract = acc_mod.extract_tables
    acc_mod.extract_tables = lambda r: (n_extract.append(1) or real_extract(r))
    try:
        e1 = RecordingEngine()
        hipporag_b200.accelerate(rag, engine=e1)
        rag.prepare_retrieval_objects()
        assert rag._b200_state["cache_hit"] is False and n_extract == [1]
        assert (tmp_path / cache.NPZ_NAME).exists() and (tmp_path / cache.META_NAME).exists()
        want = build_transition_csr(kg.n_nodes, kg.edge_src, kg.edge_dst, kg.edge_w)
        e2 = RecordingEngine()
        hipporag_b200.accelerate(rag, engine=e2)
        rag.prepare_retrieval_objects()
        assert rag._b200_state["cache_hit"] is True and n_extract == [1]            # nothing re-derived in Python
        for got in (e1.calls[0], e2.calls[0]):
            assert got[1] == kg.n_nodes
            for a, b in zip(got[2:], want):
                np.testing.assert_array_equal(a, b)
        for a, b in zip(e1.calls[1][1:], e2.calls[1][1:]):
            np.testing.assert_array_equal(a, b)
        assert rag._b200_state["facts"] == [tuple(f) for f in real_extract(rag)["facts"]]
        # cache=False never touches the directory; a changed index misses
        fp = cache.fingerprint(rag)
        assert cache.load(str(tmp_path), fp) is not None
        rag.passage_node_keys = list(rag.passage_node_keys[:-1]) + ["chunk-renamed"]
        assert cache.fingerprint(rag) != fp and cache.load(str(tmp_path), cache.fingerprint(rag)) is None
        # a corrupt file is a miss, not an error
        (tmp_path / cache.META_NAME).write_text("{not json")
        assert cache.load(str(tmp_path), fp) is None
    finally:
        acc_mod.extract_tables = real_extract
