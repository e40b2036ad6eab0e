"""The drop-in (hipporag_b200.accelerate): host glue against the reference's own object, replayed from a
recording (CPU, oracle-backed engine double), and the GPU path through a duck-typed HippoRAG (GPU box)."""
import json
import os

import numpy as np
import pytest

from oracle import ppr, retrieve


class OracleEngine:
    """Test double with Engine's interface, computing with the float64 oracle (CPU-only glue test)."""
    dim = 0

    def load_graph(self, n, src, dst, w):
        self.n = n
        self.P = ppr.transition_matrix(ppr.symmetric_weights(n, src, dst, w))[0]

    def load_graph_csr(self, n, row_ptr, col, val):
        import scipy.sparse as sp
        self.n = n
        self.P = sp.csr_matrix((np.asarray(val, np.float64), col, row_ptr), shape=(n, n))

    def load_tables(self, pv, fs, fo, cc):
        self.tb = retrieve.Tables(self.n, np.asarray(pv), np.asarray(fs), np.asarray(fo), np.asarray(cc))

    def load_embeddings(self, fe, pe):
        self.fe, self.pe, self.dim = fe, pe, pe.shape[1]

    def set_options(self, **kw):
        pass

    def stage_a(self, Q, k):
        idx = np.full((len(Q), k), -1, np.int32); sc = np.zeros((len(Q), k), np.float32); nv = np.zeros(len(Q), np.int32)
        for i, q in enumerate(Q):
            fs = retrieve.fact_scores(self.fe, q)
            top = retrieve.top_facts(fs, k)
            idx[i, :len(top)] = top; sc[i, :len(top)] = fs[top]; nv[i] = len(top)
        return idx, sc, nv

    def similarity(self, which, Q):
        E = self.fe if which == 0 else self.pe
        return np.stack([retrieve.min_max_normalize(np.dot(E, q)) for q in Q])

    def ppr(self, reset, damping=0.5, iters=0, tol=0.0):
        return ppr.ppr_power(self.P, np.asarray(reset, dtype=np.float64), damping)

    def stage_b(self, Q, kept_idx, kept_score, dpr_only, damping, pnw, link_top_k, topk, iters=0, tol=0.0):
        ids = np.full((len(Q), topk), -1, np.int32); sc = np.zeros((len(Q), topk), np.float32)
        for i, q in enumerate(Q):
            kept = [int(j) for j in kept_idx[i] if j >= 0]
            ps = retrieve.passage_scores(self.pe, q)
            if not kept:
                order = retrieve.order_desc(ps, topk); s = ps[order]
            else:
                fs = np.zeros(self.fe.shape[0]); fs[kept] = kept_score[i, :len(kept)]
                r, _ = retrieve.seed_vector(self.tb, fs, kept, ps, link_top_k, pnw)
                pi = ppr.ppr_power(self.P, r, damping)[self.tb.passage_vid]
                order = retrieve.order_desc(pi, topk); s = pi[order]
            ids[i, :len(order)] = order; sc[i, :len(order)] = s
        return ids, sc


class FakeQALLM:
    """IRCoT reasoning double: the thought depends on the question and on how many thoughts came before."""

    def infer(self, messages):
        text = messages[-1]["content"] if isinstance(messages[-1], dict) else str(messages[-1])
        q = text.rsplit("Question:", 1)[-1]
        n_prev = q.count("thought-")
        tag = "thought-%d about %s" % (n_prev, q.split("\n")[0].strip()[:40])
        return [tag + (" So the answer is: x" if n_prev >= 1 and len(q) % 2 == 0 else "")]


def test_accelerate_glue_against_reference_object(tmp_path):
    """The reference's own HippoRAG object, replayed from tests/golden/reference_rag150.npz (state after its index()
    and what its own retrieve / retrieve_ircot returned; see tests/golden/make_reference_rag.py)."""
    from tests import fake_hipporag
    fake_hipporag.install_stub_package()
    import hipporag_b200
    from hipporag.utils.misc_utils import QuerySolution
    g, rag = fake_hipporag.load_recorded_rag(str(tmp_path))
    questions = g["questions"].tolist()
    ref_docs = [[rag.passage_texts[i] for i in row] for row in g["ref_doc_ids"]]
    ref_seeds = json.loads(str(g["ref_graph_seeds"]))
    hipporag_b200.accelerate(rag, engine=OracleEngine())
    rag.ready_to_retrieve = False
    acc = rag.retrieve(questions, num_to_retrieve=20)
    assert len(acc) == len(ref_docs)
    same = 0
    for a, q, r_docs, r_scores, r_seeds in zip(acc, questions, ref_docs, g["ref_doc_scores"], ref_seeds):
        assert a.question == q and len(a.docs) == len(r_docs) == 20
        assert type(a) is QuerySolution
        overlap = len(set(a.docs) & set(r_docs)) / 20
        assert overlap >= 0.8
        assert [tuple(f) for f in a.graph_seeds] == [tuple(f) for f in r_seeds]
        if a.docs == r_docs and np.allclose(a.doc_scores, r_scores, rtol=1e-5):
            same += 1
    assert same >= len(ref_docs) // 2          # the rest differ only by the reference's set-order tie-break
    assert rag.all_retrieval_time > 0 and rag.ppr_time > 0
    # the thread-pooled filter gives the same answers as the serial one
    hipporag_b200.accelerate(rag, engine=OracleEngine(), filter_workers=4)
    rag.ready_to_retrieve = False
    par = rag.retrieve(questions, num_to_retrieve=20)
    assert [p.docs for p in par] == [a.docs for a in acc]
    # IRCoT: the batched, step-synchronous drop-in must equal the reference's serial loop (HippoRAG.py:509)
    rag.qa_llm = FakeQALLM()
    got = rag.retrieve_ircot(questions[:6], max_qa_steps=3, num_to_retrieve=10)
    want = zip(json.loads(str(g["ircot_doc_ids"])), json.loads(str(g["ircot_doc_scores"])),
               json.loads(str(g["ircot_thoughts"])))
    assert len(got) == 6
    for a, (b_ids, b_scores, b_thoughts) in zip(got, want):
        assert a.docs == [rag.passage_texts[i] for i in b_ids] and a.thoughts == b_thoughts
        np.testing.assert_allclose(a.doc_scores, b_scores)
    # the binary cache (8(f)-3): written next to graph.pickle on the first prepare, reused while the index is unchanged
    import sys as _sys
    from hipporag_b200 import cache as cache_mod
    acc_mod = _sys.modules["hipporag_b200.accelerate"]        # the module (the package re-exports the function)
    assert os.path.exists(os.path.join(rag.working_dir, cache_mod.NPZ_NAME))
    assert rag._b200_state["cache_hit"] in (True, False)
    calls = []
    real_extract = acc_mod.extract_tables
    acc_mod.extract_tables = lambda r: (calls.append(1) or real_extract(r))
    try:
        hipporag_b200.accelerate(rag, engine=OracleEngine())
        rag.ready_to_retrieve = False
        cached = rag.retrieve(questions, num_to_retrieve=20)
        assert rag._b200_state["cache_hit"] is True and calls == []          # no Python re-derivation
        assert [c.docs for c in cached] == [a.docs for a in acc]
        for c, a in zip(cached, acc):
            np.testing.assert_allclose(c.doc_scores, a.doc_scores, rtol=1e-6)   # fp32 P from the cache vs f64 edge list
        # a changed index invalidates it: one more edge -> different fingerprint -> rebuilt
        fp0 = cache_mod.fingerprint(rag)
        rag.graph.add_edges([(rag.graph.vs["name"][0], rag.graph.vs["name"][1])], attributes={"weight": [0.5]})
        assert cache_mod.fingerprint(rag) != fp0 and cache_mod.load(rag.working_dir, cache_mod.fingerprint(rag)) is None
        rag.ready_to_retrieve = False
        rag.retrieve(questions[:2], num_to_retrieve=5)
        assert rag._b200_state["cache_hit"] is False and calls == [1]
    finally:
        acc_mod.extract_tables = real_extract
    # linking_top_k is honoured, not clamped (config_utils.py:184): 10 candidates reach the filter; > 32 raises
    seen = []
    orig_filter = rag.rerank_filter
    rag.rerank_filter = lambda q, c, i, len_after_rerank=None: (seen.append(len(c)) or (i[:len_after_rerank], c[:len_after_rerank], {}))
    rag.global_config.linking_top_k = 10
    ref10 = json.loads(str(g["ref10_graph_seeds"]))                          # the reference's own retrieve
    seen.clear()
    acc10 = rag.retrieve(questions[:4], num_to_retrieve=10)
    assert seen == [10, 10, 10, 10] and len(ref10) == 4
    for a, r in zip(acc10, ref10):
        assert [tuple(f) for f in a.graph_seeds] == [tuple(f) for f in r] and len(a.graph_seeds) == 10
    rag.global_config.linking_top_k = 40
    with pytest.raises(ValueError, match="linking_top_k"):
        rag.retrieve(questions[:2], num_to_retrieve=5)
    rag.global_config.linking_top_k = 5
    rag.rerank_filter = orig_filter
    # add_synonymy_edges is wrapped: the KNN it calls is swapped for the engine's for the duration of the call only
    import sys
    ref_mod = sys.modules[type(rag).__module__]              # the module whose retrieve_knn add_synonymy_edges calls
    from hipporag_b200 import knn as knn_mod
    calls = {}

    def fake_engine_knn(query_ids, key_ids, query_vecs, key_vecs, **kw):
        calls.update(kw)
        return {}
    saved_ref_knn, saved_knn = ref_mod.retrieve_knn, knn_mod.retrieve_knn
    knn_mod.retrieve_knn = fake_engine_knn
    try:
        rag.add_synonymy_edges()
    finally:
        knn_mod.retrieve_knn = saved_knn
    assert calls.get("min_score") == rag.global_config.synonymy_edge_sim_threshold and "k" in calls
    assert ref_mod.retrieve_knn is saved_ref_knn
    # a filter that keeps nothing -> DPR fallback for every query
    rag.rerank_filter = lambda q, c, i, len_after_rerank=None: ([], [], {})
    for s in rag.retrieve(questions[:3], num_to_retrieve=5):
        assert len(s.docs) == 5 and s.graph_seeds == []


@pytest.mark.gpu
def test_accelerate_on_gpu_with_duck_typed_rag():
    from tests import fake_hipporag
    fake_hipporag.install_stub_package()
    import hipporag_b200
    from hipporag_b200 import synth
    kg = synth.make_kg(3000, 30000, seed=5)
    d = 64
    fe, pe = synth.unit_rows(kg.n_facts, d, 1), synth.unit_rows(kg.n_pass, d, 2)
    qf, qp, _ = synth.make_queries(kg, fe, pe, 10, seed=3)
    queries = [f"question {i}" for i in range(10)]
    rag = fake_hipporag.FakeRag(kg, fe, pe, qf, qp, queries)
    hipporag_b200.accelerate(rag, device=0)
    sols = rag.retrieve(queries, num_to_retrieve=25)
    P = ppr.transition_matrix(ppr.symmetric_weights(kg.n_nodes, kg.edge_src, kg.edge_dst, kg.edge_w))[0]
    tb = retrieve.Tables(kg.n_nodes, kg.passage_vid, kg.fact_subj_vid, kg.fact_obj_vid, kg.ent_chunk_count)
    for i, s in enumerate(sols):
        o = retrieve.retrieve_one(P, tb, fe, pe, qf[i], qp[i], top_k=25)
        assert s.docs == [f"passage {j}" for j in o["ids"]]
        np.testing.assert_allclose(s.doc_scores, o["scores"], rtol=5e-5)
        assert len(s.graph_seeds) == 5
    # retrieve_dpr: dense retrieval only
    for i, s in enumerate(rag.retrieve_dpr(queries, num_to_retrieve=7)):
        want = retrieve.passage_scores(pe, qp[i])
        order = retrieve.order_desc(want, 7)
        assert s.docs == [f"passage {j}" for j in order]
        np.testing.assert_allclose(s.doc_scores, want[order], atol=8e-6)
    # direct single-call forms
    ids, sc = rag.dense_passage_retrieval(queries[0])
    want = retrieve.passage_scores(pe, qp[0])
    assert ids.shape[0] == kg.n_pass and ids[0] == np.argmax(want)
    np.testing.assert_allclose(sc, want[ids], atol=5e-6)
    fsc = rag.get_fact_scores(queries[0])
    np.testing.assert_allclose(fsc, retrieve.fact_scores(fe, qf[0]), atol=5e-6)
    r = np.zeros(kg.n_nodes); r[kg.passage_vid[:5]] = 1.0; r[7] = 2.0
    ids2, sc2 = rag.run_ppr(r, 0.5)
    want2 = ppr.ppr_direct(P, r, 0.5)[kg.passage_vid]
    assert ids2.shape[0] == kg.n_pass
    np.testing.assert_allclose(sc2, want2[ids2], rtol=5e-5, atol=1e-9)


@pytest.mark.gpu
def test_synonymy_knn_through_the_wrapped_add_synonymy_edges():
    """SURVEY.md 8(f)-2: add_synonymy_edges run through accelerate() (threshold applied in the GEMM epilogue) adds the
    same synonymy edges, with the same scores, as the plain cosine top-k it replaces."""
    from tests import fake_hipporag
    fake_hipporag.install_stub_package()
    import hipporag_b200
    from hipporag_b200 import synth
    kg = synth.make_kg(3000, 30000, seed=5)
    d = 64
    fe, pe = synth.unit_rows(kg.n_facts, d, 1), synth.unit_rows(kg.n_pass, d, 2)
    qf, qp, _ = synth.make_queries(kg, fe, pe, 4, seed=3)
    rng = np.random.default_rng(0)
    base = synth.unit_rows(300, d, 9)                       # 300 clusters of near-synonyms + noise
    ent = base[rng.integers(0, 300, kg.n_ent)] + 0.04 * rng.standard_normal((kg.n_ent, d)).astype(np.float32)
    ent[5] = ent[6]                                         # exact duplicates: score 1.0, tie broken by row
    ent *= rng.uniform(0.5, 2.0, (kg.n_ent, 1)).astype(np.float32)      # the KNN normalises
    contents = [f"entity number {i}" for i in range(kg.n_ent)]
    contents[11] = "ab"                                     # too short: skipped as a query (HippoRAG.py:1000)
    contents[12] = ""                                       # empty phrase: never accepted as a neighbour (:1010)

    def run(accelerated):
        rag = fake_hipporag.FakeRag(kg, fe, pe, qf, qp, [f"q{i}" for i in range(4)])
        rag.set_entity_embeddings(ent, list(contents))
        if accelerated:
            hipporag_b200.accelerate(rag, device=0)
        rag.add_synonymy_edges()
        return rag.node_to_node_stats
    want, got = run(False), run(True)
    assert len(want) > 1000
    # membership can differ only where a score sits within fp32 noise of the 0.8 threshold
    for key in set(want) ^ set(got):
        assert abs((want.get(key) or got.get(key)) - 0.8) < 1e-5, key
    for key in set(want) & set(got):
        assert abs(want[key] - got[key]) < 1e-5
    assert fake_hipporag.retrieve_knn.__module__ == "tests.fake_hipporag"      # the swap was undone


@pytest.mark.gpu
def test_retrieve_ircot_batched_equals_the_serial_loop_on_gpu():
    """SURVEY.md 8(f)-4: the step-synchronous retrieve_ircot (every reasoning round = ONE batched stage A/B over the
    queries still active) returns what the reference's per-query loop (HippoRAG.py:509-558, restated below on top of
    single-query retrieve calls) returns: same documents, scores and thoughts."""
    from tests import fake_hipporag
    fake_hipporag.install_stub_package()
    import types
    import hipporag_b200
    from hipporag.utils.misc_utils import QuerySolution
    from hipporag.utils.qa_utils import reason_step
    from hipporag_b200 import synth
    kg = synth.make_kg(3000, 30000, seed=8)
    d = 64
    fe, pe = synth.unit_rows(kg.n_facts, d, 1), synth.unit_rows(kg.n_pass, d, 2)
    nq, steps, topn = 12, 3, 10
    queries = [f"question {i}" for i in range(nq)]
    # every string that can become a query (a question or a thought) has a deterministic embedding pair
    texts = list(queries)
    for i in range(nq):
        for n_prev in range(steps):
            texts.append(f"thought-{n_prev} about question {i}")
    rng = np.random.default_rng(0)
    j = rng.integers(0, kg.n_facts, len(texts))
    qf = fe[j] + 0.3 * synth.unit_rows(len(texts), d, 5)
    qp = pe[kg.fact_passage[j]] + 0.3 * synth.unit_rows(len(texts), d, 6)
    qf /= np.linalg.norm(qf, axis=1, keepdims=True)
    qp /= np.linalg.norm(qp, axis=1, keepdims=True)

    class QALLM:                      # thought depends on the question and on how many thoughts came before
        def infer(self, messages):
            text = messages if isinstance(messages, str) else str(messages)
            q = text.rsplit("Question:", 1)[-1]
            name = q.split("\n")[0].strip()
            n_prev = q.count("thought-")
            idx = int(name.split()[-1])
            return [f"thought-{n_prev} about {name}" + (" So the answer is: x" if n_prev >= 1 and idx % 3 == 0 else "")]

    def make():
        rag = fake_hipporag.FakeRag(kg, fe, pe, qf, qp, texts)
        rag.global_config.dataset = "musique"
        rag.prompt_template_manager = types.SimpleNamespace(is_template_name_valid=lambda name: True,
                                                            render=lambda name, prompt_user: prompt_user)
        rag.qa_llm = QALLM()
        hipporag_b200.accelerate(rag, device=0)
        return rag
    rag = make()
    got = rag.retrieve_ircot(queries, max_qa_steps=steps, num_to_retrieve=topn)
    # the reference's loop, one query at a time, on single-query retrieve calls of the same engine
    want = []
    for query in queries:
        step = rag.retrieve([query], num_to_retrieve=topn)[0]
        merged = dict(zip(step.docs, np.asarray(step.doc_scores).tolist()))
        thoughts = []
        for _ in range(1, steps):
            ranked = sorted(merged, key=merged.get, reverse=True)
            thought = reason_step("musique", rag.prompt_template_manager, query, ranked[:topn], thoughts, rag.qa_llm)
            thoughts.append(thought)
            if "So the answer is:" in thought:
                break
            step = rag.retrieve([thought], num_to_retrieve=topn)[0]
            for doc, score in zip(step.docs, np.asarray(step.doc_scores).tolist()):
                merged[doc] = max(merged.get(doc, float("-inf")), score)
        items = sorted(merged.items(), key=lambda it: it[1], reverse=True)
        want.append(([dd for dd, _ in items], np.asarray([sc for _, sc in items]), thoughts))
    assert len(got) == nq and all(isinstance(g, QuerySolution) for g in got)
    for g, (docs, scores, thoughts) in zip(got, want):
        assert g.thoughts == thoughts
        assert set(g.docs) == set(docs) and len(g.docs) == len(docs)
        # a batch of 12 takes the fp32 solver at width 16, a single query at width 4: same answers to fp32 round-off
        np.testing.assert_allclose(np.sort(np.asarray(g.doc_scores))[::-1], np.sort(scores)[::-1], rtol=2e-5)
    assert any(len(t) == 1 for _, _, t in want) or any(len(t) == 2 for _, _, t in want)
