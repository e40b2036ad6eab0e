"""Generates ``tests/golden/reference_rag150.npz``: a ``HippoRAG`` object as the reference's own
unmodified ``index()`` leaves it on the first 150 MuSiQue passages (64-d md5-seeded mock embeddings,
identity recognition-memory filter), and what the reference's own methods returned on it.

Run with a checkout of the reference:   PYTHONHASHSEED=0 python tests/golden/make_reference_rag.py <reference checkout>

``tests/fake_hipporag.RecordedRag`` rebuilds the object from the recorded state (graph, stores, chunk
counts, config; node keys are md5 ids of the texts, so only the texts and the positions of the keys are
kept); ``tests/test_accelerate.py`` and ``tests/test_host_logic.py`` hold the drop-in to the
recorded outputs:

* ``harness_*``: ``oracle.ref_harness.extract_tables`` on the reference object;
* ``ref_*``: ``HippoRAG.retrieve`` of the first 12 MuSiQue questions (top 20);
* ``ircot_*``: ``HippoRAG.retrieve_ircot`` (the reference's serial loop) of the first 6 questions,
  3 steps, top 10, over the drop-in's ``retrieve`` with the float64 oracle engine
  (``tests.test_accelerate.OracleEngine``) and ``tests.test_accelerate.FakeQALLM``;
* ``ref10_graph_seeds``: ``HippoRAG.retrieve`` of the first 4 questions with ``linking_top_k = 10``.

Embeddings are not stored: the texts are, and the mock embedder regenerates them from their md5 seeds.
"""
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import ref_harness as H  # noqa: E402

N_DOCS, DIM, N_Q = 150, 64, 12


def main(reference_root):
    H.REFERENCE_ROOT = os.path.abspath(reference_root)
    H.install_stubs()
    from hipporag.prompts.linking import get_query_instruction
    import hipporag_b200
    from tests.test_accelerate import FakeQALLM, OracleEngine

    rag = H.build_reference_rag(tempfile.mkdtemp(prefix="hrag_rec_"), N_DOCS, DIM)
    questions = H.musique_questions(N_Q)
    tables = H.extract_tables(rag)                       # runs prepare_retrieval_objects

    # the state the drop-in reads, before any retrieval touches the object
    from hipporag.utils.misc_utils import compute_mdhash_id
    ent_keys = list(rag.entity_embedding_store.get_all_ids())
    ent_texts = [rag.entity_embedding_store.get_row(k)["content"] for k in ent_keys]
    passage_texts = [rag.chunk_embedding_store.get_row(k)["content"] for k in rag.passage_node_keys]
    # keys are md5 ids of the texts: stored as positions, rebuilt by RecordedRag
    assert ent_keys == [compute_mdhash_id(t, prefix="entity-") for t in ent_texts]
    assert rag.passage_node_keys == [compute_mdhash_id(t, prefix="chunk-") for t in passage_texts]
    assert rag.fact_node_keys == [compute_mdhash_id(t, prefix="fact-") for t in tables["fact_texts"]]
    key_pos = {k: i for i, k in enumerate(ent_keys + rag.passage_node_keys)}
    vertex_key = [key_pos[n] for n in rag.graph.vs["name"]]
    chunk_keys = sorted(rag.ent_node_to_chunk_ids)
    cfg = rag.global_config
    config = dict(retrieval_top_k=cfg.retrieval_top_k, linking_top_k=cfg.linking_top_k, damping=cfg.damping,
                  passage_node_weight=cfg.passage_node_weight, dataset=cfg.dataset,
                  synonymy_edge_topk=cfg.synonymy_edge_topk,
                  synonymy_edge_sim_threshold=cfg.synonymy_edge_sim_threshold,
                  synonymy_edge_query_batch_size=cfg.synonymy_edge_query_batch_size,
                  synonymy_edge_key_batch_size=cfg.synonymy_edge_key_batch_size)
    pidx = {t: i for i, t in enumerate(passage_texts)}

    def doc_ids(sol):
        return np.array([pidx[d] for d in sol.docs], dtype=np.int32)

    ref = rag.retrieve(questions, num_to_retrieve=20)
    # the object goes through the steps test_accelerate_glue_against_reference_object takes before its IRCoT
    # check: the second prepare reads the index cache the first one wrote
    for workers in (1, 4):
        hipporag_b200.accelerate(rag, engine=OracleEngine(), filter_workers=workers)
        rag.ready_to_retrieve = False
        rag.retrieve(questions, num_to_retrieve=20)
    rag.qa_llm = FakeQALLM()
    ircot = type(rag).retrieve_ircot(rag, questions[:6], max_qa_steps=3, num_to_retrieve=10)
    rag.global_config.linking_top_k = 10
    ref10 = type(rag).retrieve(rag, questions[:4], num_to_retrieve=10)

    out = dict(
        dim=np.int32(DIM), config=np.array(json.dumps(config)), questions=np.array(questions),
        query_instruction_fact=np.array(get_query_instruction("query_to_fact")),
        query_instruction_passage=np.array(get_query_instruction("query_to_passage")),
        vertex_key=np.array(vertex_key, dtype=np.int32), edge_src=tables["edge_src"], edge_dst=tables["edge_dst"],
        edge_w=tables["edge_w"], passage_texts=np.array(passage_texts), fact_texts=np.array(tables["fact_texts"]),
        entity_texts=np.array(ent_texts),
        chunk_count_entity=np.array([ent_keys.index(k) for k in chunk_keys], dtype=np.int32),
        chunk_counts=np.array([len(rag.ent_node_to_chunk_ids[k]) for k in chunk_keys], dtype=np.int32),
        harness_n_nodes=np.int64(tables["n_nodes"]), harness_passage_vid=tables["passage_vid"],
        harness_fact_subj_vid=tables["fact_subj_vid"], harness_fact_obj_vid=tables["fact_obj_vid"],
        harness_ent_chunk_count=tables["ent_chunk_count"],
        ref_doc_ids=np.stack([doc_ids(s) for s in ref]),
        ref_doc_scores=np.stack([np.asarray(s.doc_scores, dtype=np.float64) for s in ref]),
        ref_graph_seeds=np.array(json.dumps([[list(f) for f in s.graph_seeds] for s in ref])),
        ircot_doc_ids=np.array(json.dumps([doc_ids(s).tolist() for s in ircot])),
        ircot_doc_scores=np.array(json.dumps([np.asarray(s.doc_scores, dtype=np.float64).tolist() for s in ircot])),
        ircot_thoughts=np.array(json.dumps([list(s.thoughts) for s in ircot])),
        ref10_graph_seeds=np.array(json.dumps([[list(f) for f in s.graph_seeds] for s in ref10])),
    )
    # self-check: the texts regenerate the embeddings the reference used
    emb = H.MockEmbeddingModel(DIM)
    assert np.array_equal(emb.batch_encode(passage_texts), rag.passage_embeddings)
    assert np.array_equal(emb.batch_encode(list(tables["fact_texts"])), rag.fact_embeddings)
    path = os.path.join(ROOT, "tests", "golden", "reference_rag150.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
