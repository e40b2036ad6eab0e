"""A duck-typed stand-in for the reference's ``HippoRAG`` object (and the two helpers of
``hipporag.utils.misc_utils`` the drop-in imports), for boxes where /root/reference is absent.
Only what ``hipporag_b200.accelerate`` touches is modelled."""
import hashlib
import json
import os
import sys
import types
from dataclasses import dataclass
from typing import Any, List

import numpy as np

from oracle.fake_igraph import Graph


def install_stub_package():
    if "hipporag" in sys.modules and not getattr(sys.modules["hipporag"], "__stub__", False):
        return                                   # the real reference package is importable
    pkg = types.ModuleType("hipporag"); pkg.__path__ = []; pkg.__stub__ = True
    utils = types.ModuleType("hipporag.utils"); utils.__path__ = []
    misc = types.ModuleType("hipporag.utils.misc_utils")

    @dataclass
    class QuerySolution:
        question: str
        docs: List[str]
        doc_scores: Any = None
        answer: str = None
        gold_answers: List[str] = None
        gold_docs: List[str] = None
        doc_metadata: Any = None
        graph_seeds: Any = None
        thoughts: Any = None

    def compute_mdhash_id(content: str, prefix: str = "") -> str:
        return prefix + hashlib.md5(content.encode()).hexdigest()

    misc.QuerySolution, misc.compute_mdhash_id = QuerySolution, compute_mdhash_id
    QuerySolution.__dataclass_fields__  # (dataclass) -- `thoughts` is set as an attribute by retrieve_ircot
    qa = types.ModuleType("hipporag.utils.qa_utils")

    def reason_step(dataset, prompt_template_manager, query, passages, thoughts, llm_client):
        """qa_utils.py:31-50: render the IRCoT prompt from the passages + question + thoughts, one LLM call."""
        prompt_user = "".join(f"{p}\n\n" for p in passages) + f"Question: {query}\nThought:" + " ".join(thoughts)
        return llm_client.infer(prompt_template_manager.render(name=f"ircot_{dataset}", prompt_user=prompt_user))[0]

    qa.reason_step = reason_step
    sys.modules.update({"hipporag": pkg, "hipporag.utils": utils, "hipporag.utils.misc_utils": misc,
                        "hipporag.utils.qa_utils": qa})


def retrieve_knn(query_ids, key_ids, query_vecs, key_vecs, k=2047, query_batch_size=1000, key_batch_size=10000):
    """The contract of ``hipporag.utils.embed_utils.retrieve_knn`` (embed_utils.py:6-94) in plain numpy: cosine
    top-k of every query against all keys, best first -- what ``add_synonymy_edges`` calls through the module
    global of the same name (HippoRAG.py:35, :986-992)."""
    if len(key_vecs) == 0:
        return {}
    q = np.asarray(query_vecs, dtype=np.float32)
    kv = np.asarray(key_vecs, dtype=np.float32)
    q = q / np.maximum(np.linalg.norm(q, axis=1, keepdims=True), 1e-12)
    kv = kv / np.maximum(np.linalg.norm(kv, axis=1, keepdims=True), 1e-12)
    out = {}
    for i0 in range(0, len(q), 256):
        S = q[i0:i0 + 256] @ kv.T
        for r in range(S.shape[0]):
            order = np.lexsort((np.arange(S.shape[1]), -S[r]))[:min(k, S.shape[1])]
            out[query_ids[i0 + r]] = ([key_ids[j] for j in order], S[r, order].tolist())
    return out


class _Store:
    def __init__(self, keys, contents):
        self.rows = {k: {"hash_id": k, "content": c} for k, c in zip(keys, contents)}

    def get_rows(self, keys):
        return {k: self.rows[k] for k in keys}

    def get_row(self, key):
        return self.rows[key]

    def get_all_id_to_rows(self):
        return dict(self.rows)

    def get_embeddings(self, keys):
        return self.emb[[self.index[k] for k in keys]]


@dataclass
class _Result:
    query: str
    docs: list
    scores: Any
    doc_metadata: list
    graph_seeds: list


class FakeRag:
    """Graph + stores + embeddings laid out like a prepared HippoRAG object."""

    def __init__(self, kg, fact_emb, passage_emb, q_fact, q_pass, queries):
        from hipporag.utils.misc_utils import compute_mdhash_id
        self.global_config = types.SimpleNamespace(retrieval_top_k=200, linking_top_k=5, damping=0.5,
                                                   passage_node_weight=0.05)
        ent_names = [f"e{i}" for i in range(kg.n_ent)]
        self.entity_keys = [compute_mdhash_id(n, "entity-") for n in ent_names]
        self.passage_node_keys = [compute_mdhash_id(f"passage {i}", "chunk-") for i in range(kg.n_pass)]
        g = Graph(directed=False)
        g.add_vertices(kg.n_nodes, attributes={"name": self.entity_keys + self.passage_node_keys})
        g.add_edges(list(zip(kg.edge_src.tolist(), kg.edge_dst.tolist())), attributes={"weight": kg.edge_w.tolist()})
        self.graph = g
        self.fact_node_keys = [f"fact-{i}" for i in range(kg.n_facts)]
        facts = [str((ent_names[s], "rel", ent_names[o])) for s, o in zip(kg.fact_subj_vid, kg.fact_obj_vid)]
        self.fact_embedding_store = _Store(self.fact_node_keys, facts)
        self.chunk_embedding_store = _Store(self.passage_node_keys, [f"passage {i}" for i in range(kg.n_pass)])
        self.chunk_metadata = {}
        self._fact_emb, self._passage_emb = fact_emb, passage_emb
        self._q = {"triple": dict(zip(queries, q_fact)), "passage": dict(zip(queries, q_pass))}
        self._kg = kg
        self.ready_to_retrieve = False
        self.ppr_time = self.rerank_time = self.all_retrieval_time = 0.0
        self.rerank_filter = lambda q, cands, idxs, len_after_rerank=None: (idxs[:len_after_rerank],
                                                                          cands[:len_after_rerank], {})

    def prepare_retrieval_objects(self):
        self.node_name_to_vertex_idx = {n: i for i, n in enumerate(self.graph.vs["name"])}
        self.passage_node_idxs = [self.node_name_to_vertex_idx[k] for k in self.passage_node_keys]
        self.fact_embeddings, self.passage_embeddings = self._fact_emb, self._passage_emb
        self.ent_node_to_chunk_ids = {self.entity_keys[v]: set(range(int(c)))
                                      for v, c in enumerate(self._kg.ent_chunk_count[:self._kg.n_ent]) if c > 0}
        self.query_to_embedding = {"triple": {}, "passage": {}}
        self.ready_to_retrieve = True

    def get_query_embeddings(self, queries):
        for q in queries:
            for kind in ("triple", "passage"):
                self.query_to_embedding[kind][q] = self._q[kind][q]

    def _build_retrieval_result(self, query, ids, scores, num_to_retrieve, graph_seeds=None):
        keys = [self.passage_node_keys[i] for i in ids[:num_to_retrieve]]
        return _Result(query, [self.chunk_embedding_store.get_row(k)["content"] for k in keys],
                       np.asarray(scores[:num_to_retrieve]), [{} for _ in keys], graph_seeds or [])

    def set_entity_embeddings(self, emb, contents=None):
        """Entity store for the synonymy KNN (HippoRAG.py:980-984)."""
        contents = contents or [f"entity number {i}" for i in range(len(self.entity_keys))]
        st = _Store(self.entity_keys, contents)
        st.emb = np.asarray(emb, dtype=np.float32)
        st.index = {k: i for i, k in enumerate(self.entity_keys)}
        self.entity_embedding_store = st
        self.global_config.synonymy_edge_topk = 2047
        self.global_config.synonymy_edge_sim_threshold = 0.8
        self.global_config.synonymy_edge_query_batch_size = 1000
        self.global_config.synonymy_edge_key_batch_size = 10000
        self.node_to_node_stats = {}

    def add_synonymy_edges(self):
        """The consumer of the KNN exactly as ``HippoRAG.add_synonymy_edges`` walks it (HippoRAG.py:980-1018)."""
        import re
        self.entity_id_to_row = self.entity_embedding_store.get_all_id_to_rows()
        entity_node_keys = list(self.entity_id_to_row.keys())
        entity_embs = self.entity_embedding_store.get_embeddings(entity_node_keys)
        knn = retrieve_knn(query_ids=entity_node_keys, key_ids=entity_node_keys, query_vecs=entity_embs,
                           key_vecs=entity_embs, k=self.global_config.synonymy_edge_topk,
                           query_batch_size=self.global_config.synonymy_edge_query_batch_size,
                           key_batch_size=self.global_config.synonymy_edge_key_batch_size)
        for node_key in knn.keys():
            entity = self.entity_id_to_row[node_key]["content"]
            if len(re.sub('[^A-Za-z0-9]', '', entity)) > 2:
                nns = knn[node_key]
                num_nns = 0
                for nn, score in zip(nns[0], nns[1]):
                    if score < self.global_config.synonymy_edge_sim_threshold or num_nns > 100:
                        break
                    nn_phrase = self.entity_id_to_row[nn]["content"]
                    if nn != node_key and nn_phrase != '':
                        self.node_to_node_stats[(node_key, nn)] = score
                        num_nns += 1

    def index(self, docs):
        pass

    def delete(self, docs):
        self.ready_to_retrieve = False


class RecordedRag(FakeRag):
    """The reference's own ``HippoRAG`` object as its ``index()`` left it, rebuilt from the recording
    ``tests/golden/reference_rag150.npz`` (``tests/golden/make_reference_rag.py``): graph, stores,
    ``ent_node_to_chunk_ids`` and config as recorded; embeddings regenerated from the stored texts by the
    md5-seeded mock embedder the recording was made with.  ``prepare_retrieval_objects``,
    ``get_query_embeddings`` and the IRCoT prompt follow HippoRAG.py:1287-1389, :1391-1425 and qa_utils.py:31-50."""

    def __init__(self, g, working_dir):
        from hipporag.utils.misc_utils import compute_mdhash_id
        from oracle.ref_harness import MockEmbeddingModel, identity_filter
        self.global_config = types.SimpleNamespace(**json.loads(str(g["config"])))
        self.working_dir = working_dir
        self.passage_texts, self.fact_texts = g["passage_texts"].tolist(), g["fact_texts"].tolist()
        ent_texts = g["entity_texts"].tolist()
        self.passage_node_keys = [compute_mdhash_id(t, prefix="chunk-") for t in self.passage_texts]
        self.fact_node_keys = [compute_mdhash_id(t, prefix="fact-") for t in self.fact_texts]
        self.entity_keys = [compute_mdhash_id(t, prefix="entity-") for t in ent_texts]
        names = [(self.entity_keys + self.passage_node_keys)[i] for i in g["vertex_key"]]
        graph = Graph(directed=False)
        graph.add_vertices(len(names), attributes={"name": names})
        graph.add_edges(list(zip(g["edge_src"].tolist(), g["edge_dst"].tolist())),
                        attributes={"weight": g["edge_w"].tolist()})
        self.graph = graph
        self.fact_embedding_store = _Store(self.fact_node_keys, self.fact_texts)
        self.chunk_embedding_store = _Store(self.passage_node_keys, self.passage_texts)
        self.ent_node_to_chunk_ids = {self.entity_keys[i]: set(range(int(c)))
                                      for i, c in zip(g["chunk_count_entity"], g["chunk_counts"])}
        self.embedding_model = MockEmbeddingModel(int(g["dim"]))
        self._instruction = {"triple": str(g["query_instruction_fact"]), "passage": str(g["query_instruction_passage"])}
        self.entity_embedding_store = _Store(self.entity_keys, ent_texts)
        self.entity_embedding_store.emb = self.embedding_model.batch_encode(ent_texts)
        self.entity_embedding_store.index = {k: i for i, k in enumerate(self.entity_keys)}
        self.node_to_node_stats = {}
        self.prompt_template_manager = types.SimpleNamespace(
            is_template_name_valid=lambda name: True,
            render=lambda name, prompt_user: [{"role": "user", "content": prompt_user}])
        self.chunk_metadata = {}
        self.ready_to_retrieve = False
        self.ppr_time = self.rerank_time = self.all_retrieval_time = 0.0
        self.rerank_filter = identity_filter

    def prepare_retrieval_objects(self):
        self.query_to_embedding = {"triple": {}, "passage": {}}
        self.node_name_to_vertex_idx = {n: i for i, n in enumerate(self.graph.vs["name"])}
        self.passage_node_idxs = [self.node_name_to_vertex_idx[k] for k in self.passage_node_keys]
        self.passage_embeddings = self.embedding_model.batch_encode(self.passage_texts)
        self.fact_embeddings = self.embedding_model.batch_encode(self.fact_texts)
        self.ready_to_retrieve = True

    def get_query_embeddings(self, queries):
        new = [q for q in queries if q not in self.query_to_embedding["triple"]
               or q not in self.query_to_embedding["passage"]]
        for kind in ("triple", "passage") if new else ():
            emb = self.embedding_model.batch_encode(new, instruction=self._instruction[kind])
            self.query_to_embedding[kind].update(zip(new, emb))


def load_recorded_rag(working_dir):
    """-> (the recording's arrays, a RecordedRag built from them that keeps its index cache in working_dir)."""
    g = dict(np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_rag150.npz")))
    return g, RecordedRag(g, working_dir)
