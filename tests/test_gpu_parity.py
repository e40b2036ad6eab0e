"""GPU parity tests: the CUDA path (through the C ABI) against the float64 oracle on the same
seeded inputs.  Tolerances live in tests/util.py (top-k identical up to oracle near-ties,
scores within 1e-5 absolute AND 2e-5 relative)."""
import numpy as np
import pytest

from oracle import ppr, retrieve
from tests.util import ATOL, RTOL, assert_topk_matches

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hb():
    import hipporag_b200
    return hipporag_b200


def _engine_for_graph(hb, n, src, dst, w):
    e = hb.Engine(0)
    e.load_graph(n, src, dst, w)
    return e


def _oracle_P(n, src, dst, w):
    return ppr.transition_matrix(ppr.symmetric_weights(n, src, dst, w))[0]


# ------------------------------------------------------------------------------ K1: PPR
@pytest.mark.parametrize("method", ["power", "chebyshev"])
def test_ppr_closed_forms(hb, method):
    m = hb.PPR_POWER if method == "power" else hb.PPR_CHEBYSHEV
    iters = 40 if method == "power" else 24
    # two nodes, one edge -> (2/3, 1/3)
    e = _engine_for_graph(hb, 2, [0], [1], [1.0])
    e.set_options(ppr_method=m, ppr_iters=iters)
    np.testing.assert_allclose(e.ppr(np.array([1.0, 0.0])), [2 / 3, 1 / 3], atol=2e-7)
    # star: hub 1/(1-a^2), leaves a/3 of it
    e = _engine_for_graph(hb, 4, [0, 0, 0], [1, 2, 3], [1, 1, 1])
    e.set_options(ppr_method=m, ppr_iters=iters)
    hub = 1 / 0.75
    leaf = 0.5 / 3 * hub
    tot = hub + 3 * leaf
    np.testing.assert_allclose(e.ppr(np.array([1.0, 0, 0, 0])), [hub / tot] + [leaf / tot] * 3, atol=2e-7)
    # isolated seed keeps all mass; isolated non-seed gets none; NaN / negative reset entries -> 0
    e = _engine_for_graph(hb, 4, [0], [1], [1.0])
    e.set_options(ppr_method=m, ppr_iters=iters)
    np.testing.assert_allclose(e.ppr(np.array([0.0, 0, 1, 0])), [0, 0, 1, 0], atol=1e-7)
    out = e.ppr(np.array([1.0, np.nan, 0, -5.0]))
    assert out[2] == 0 and out[3] == 0
    np.testing.assert_allclose(out[:2], [2 / 3, 1 / 3], atol=2e-7)


@pytest.mark.parametrize("method,iters", [("power", 30), ("chebyshev", 16)])
@pytest.mark.parametrize("batch", [1, 5, 16, 37])
def test_ppr_random_graph_vs_oracle(hb, method, iters, batch):
    from hipporag_b200 import synth
    kg = synth.make_kg(20_000, 200_000, seed=3)
    n = kg.n_nodes
    P = _oracle_P(n, kg.edge_src, kg.edge_dst, kg.edge_w)
    rng = np.random.default_rng(batch)
    R = np.zeros((batch, n), dtype=np.float32)
    R[:, kg.passage_vid] = 0.05 * rng.random((batch, kg.n_pass), dtype=np.float32)
    for b in range(batch):
        R[b, rng.integers(0, kg.n_ent, 5)] = rng.random(5, dtype=np.float32)
    R[0, n - kg.n_pass - 1] = 0.7          # mass on an isolated entity (a sink)
    e = _engine_for_graph(hb, n, kg.edge_src, kg.edge_dst, kg.edge_w)
    e.set_options(ppr_method=hb.PPR_POWER if method == "power" else hb.PPR_CHEBYSHEV, ppr_iters=iters,
                  ppr_batch=16)
    got = e.ppr(R)
    want = ppr.ppr_batch_power(P, R.T.astype(np.float64), 0.5).T
    np.testing.assert_allclose(got.sum(axis=1), 1.0, atol=1e-5)
    scale = want.max(axis=1, keepdims=True)
    assert np.max(np.abs(got - want) / scale) < RTOL
    assert np.max(np.abs(got - want)) < ATOL
    big = want > 1e-3 * scale
    assert np.max(np.abs(got - want)[big] / want[big]) < 5 * RTOL


def test_ppr_long_rows_hub(hb):
    # hub of degree 5000 (> long-row threshold 256, 20 segments) + a random tail: exercises the
    # segmented path; weights vary so the order of summation matters at the 1e-7 level only
    n = 6000
    rng = np.random.default_rng(0)
    src = np.concatenate([np.zeros(5000, dtype=np.int64), rng.integers(1, n, 8000)])
    dst = np.concatenate([np.arange(1, 5001), rng.integers(1, n, 8000)])
    keep = src != dst
    src, dst = src[keep], dst[keep]
    w = rng.random(src.shape[0]) + 0.5
    P = _oracle_P(n, src, dst, w)
    R = rng.random((7, n), dtype=np.float32) * (rng.random((7, n)) < 0.01)
    R[:, 0] += 0.5
    e = _engine_for_graph(hb, n, src, dst, w)
    for m, it in ((hb.PPR_POWER, 30), (hb.PPR_CHEBYSHEV, 16)):
        e.set_options(ppr_method=m, ppr_iters=it, ppr_batch=8)
        got = e.ppr(R)
        want = ppr.ppr_batch_power(P, R.T.astype(np.float64), 0.5).T
        assert np.max(np.abs(got - want) / want.max(axis=1, keepdims=True)) < RTOL


@pytest.mark.parametrize("batch", [3, 32, 45])
def test_ppr_mixed_precision_vs_oracle(hb, batch):
    """fp16 state + one fp32 refinement step must be as accurate as the all-fp32 solver."""
    from hipporag_b200 import synth
    kg = synth.make_kg(20_000, 200_000, seed=3)
    n = kg.n_nodes
    P = _oracle_P(n, kg.edge_src, kg.edge_dst, kg.edge_w)
    rng = np.random.default_rng(batch)
    R = np.zeros((batch, n), dtype=np.float32)
    R[:, kg.passage_vid] = 0.05 * rng.random((batch, kg.n_pass), dtype=np.float32)
    for b in range(batch):
        R[b, rng.integers(0, kg.n_ent, 5)] = rng.random(5, dtype=np.float32)
    R[0, n - kg.n_pass - 1] = 0.7          # mass on an isolated entity
    R[1] *= 1e-3                           # a column with a very different scale
    e = _engine_for_graph(hb, n, kg.edge_src, kg.edge_dst, kg.edge_w)
    e.set_options(ppr_precision=hb.PPR_MIXED)
    got = e.ppr(R)
    want = ppr.ppr_batch_power(P, R.T.astype(np.float64), 0.5).T
    np.testing.assert_allclose(got.sum(axis=1), 1.0, atol=1e-5)
    scale = want.max(axis=1, keepdims=True)
    assert np.max(np.abs(got - want) / scale) < RTOL
    big = want > 1e-3 * scale
    assert np.max(np.abs(got - want)[big] / want[big]) < 5 * RTOL
    st = e.stats()
    if batch > 16:      # batches of <= 16 reset vectors run the fp32 solver at their own width (same gate as stage B)
        assert st["ppr_columns"] == 32 * st["ppr_sweeps"]
        assert 0.0 < st["ppr_residual"] < 5e-3 and st["ppr_error_bound"] < 1e-5
    else:
        assert st["ppr_columns"] < 32 * st["ppr_sweeps"]


def test_ppr_mixed_long_rows_and_closed_form(hb):
    n = 6000
    rng = np.random.default_rng(0)
    src = np.concatenate([np.zeros(5000, dtype=np.int64), rng.integers(1, n, 8000)])
    dst = np.concatenate([np.arange(1, 5001), rng.integers(1, n, 8000)])
    keep = src != dst
    src, dst = src[keep], dst[keep]
    w = rng.random(src.shape[0]) + 0.5
    P = _oracle_P(n, src, dst, w)
    R = rng.random((20, n), dtype=np.float32) * (rng.random((20, n)) < 0.01)
    R[:, 0] += 0.5
    e = _engine_for_graph(hb, n, src, dst, w)
    e.set_options(ppr_precision=hb.PPR_MIXED)
    got = e.ppr(R)
    assert e.stats()["ppr_columns"] == 32 * e.stats()["ppr_sweeps"]       # the fp16 solver ran (batch > 16)
    want = ppr.ppr_batch_power(P, R.T.astype(np.float64), 0.5).T
    assert np.max(np.abs(got - want) / want.max(axis=1, keepdims=True)) < RTOL
    e2 = _engine_for_graph(hb, 2, [0], [1], [1.0])
    e2.set_options(ppr_precision=hb.PPR_MIXED)
    out = e2.ppr(np.tile(np.array([[1.0, 0.0]], np.float32), (17, 1)))
    np.testing.assert_allclose(out, np.tile([[2 / 3, 1 / 3]], (17, 1)), atol=2e-6)


@pytest.mark.parametrize("damping", [0.5, 0.85])
@pytest.mark.parametrize("batch", [5, 40])
def test_ppr_sweep_counts_follow_damping(hb, damping, batch):
    """config_utils.py:192 makes damping configurable; PRPACK converges whatever it is.  The sweep counts are
    derived from damping (Chebyshev rate a / (1 + sqrt(1 - a^2))), so accuracy must not depend on it."""
    from hipporag_b200 import synth
    kg = synth.make_kg(20_000, 200_000, seed=4)
    n = kg.n_nodes
    P = _oracle_P(n, kg.edge_src, kg.edge_dst, kg.edge_w)
    rng = np.random.default_rng(batch)
    R = np.zeros((batch, n), dtype=np.float32)
    R[:, kg.passage_vid] = 0.05 * rng.random((batch, kg.n_pass), dtype=np.float32)
    for b in range(batch):
        R[b, rng.integers(0, kg.n_ent, 5)] = rng.random(5, dtype=np.float32)
    e = _engine_for_graph(hb, n, kg.edge_src, kg.edge_dst, kg.edge_w)
    got = e.ppr(R, damping=damping)
    want = ppr.ppr_batch_power(P, R.T.astype(np.float64), damping).T
    scale = want.max(axis=1, keepdims=True)
    assert np.max(np.abs(got - want) / scale) < RTOL
    assert np.max(np.abs(got - want)) < ATOL
    st = e.stats()
    sweeps_per_solve = st["ppr_sweeps"] / -(-batch // (32 if st["ppr_columns"] == 32 * st["ppr_sweeps"] else 16))
    if damping == 0.5:
        assert sweeps_per_solve == (16 if batch > 16 else 14)
    else:
        assert sweeps_per_solve >= 30          # 0.557^k <= 1e-8 needs 32 fp32 sweeps
    # a pinned, far too small sweep count with an explicit tolerance must fail loudly (mixed solver only)
    if batch > 16 and damping == 0.5:
        with pytest.raises(hb.HragError, match="misses tol"):
            e.ppr(R, damping=damping, iters=2, tol=1e-6)
        got2 = e.ppr(R, damping=damping, iters=10, tol=1e-6)      # generous pin: passes and stays accurate
        assert np.max(np.abs(got2 - want) / scale) < RTOL


def test_retrieve_musique1k_mixed_precision(hb, golden, c1):
    g = golden
    c1.engine.set_options(ppr_precision=hb.PPR_MIXED)
    try:
        ids, scores, _, _ = c1.retrieve(g["q_fact"], g["q_pass"], topk=200)
    finally:
        c1.engine.set_options(ppr_precision=hb.PPR_FP32)
    for q in range(g["q_fact"].shape[0]):
        o = retrieve.retrieve_one(g["P"], g["tables"], g["fact_emb"], g["passage_emb"], g["q_fact"][q], g["q_pass"][q],
                                  top_k=None)
        full = np.empty(len(o["ids"]))
        full[o["ids"]] = o["scores"]
        assert_topk_matches(ids[q], scores[q], full, 200, what=f"query {q} (mixed)")


@pytest.mark.parametrize("width", [4, 8, 16, 32, 64])
def test_ppr_every_batch_width(hb, width):
    from hipporag_b200 import synth
    kg = synth.make_kg(5_000, 50_000, seed=1)
    n = kg.n_nodes
    P = _oracle_P(n, kg.edge_src, kg.edge_dst, kg.edge_w)
    R = np.random.default_rng(width).random((width, n), dtype=np.float32)
    e = _engine_for_graph(hb, n, kg.edge_src, kg.edge_dst, kg.edge_w)
    e.set_options(ppr_iters=16, ppr_batch=width)
    got = e.ppr(R)
    want = ppr.ppr_batch_power(P, R.T.astype(np.float64), 0.5).T
    assert np.max(np.abs(got - want) / want.max(axis=1, keepdims=True)) < RTOL


def test_library_graph_ingest_matches_scipy_path(hb):
    """hrag_load_graph_coo (C++ ingest) and build_transition_csr (scipy) must give the same operator."""
    from hipporag_b200 import synth
    kg = synth.make_kg(8_000, 80_000, seed=9)
    w = kg.edge_w.copy()
    w[::97] = 0.0                                   # dropped edges
    w[5::101] = -1.0
    R = np.random.default_rng(1).random((5, kg.n_nodes), dtype=np.float32)
    e1 = hb.Engine(0)
    e1.load_graph(kg.n_nodes, kg.edge_src, kg.edge_dst, w)
    e2 = hb.Engine(0)
    e2.load_graph_csr(kg.n_nodes, *hb.build_transition_csr(kg.n_nodes, kg.edge_src, kg.edge_dst, w))
    for e in (e1, e2):
        e.set_options(ppr_precision=hb.PPR_FP32)
    a, b = e1.ppr(R), e2.ppr(R)
    np.testing.assert_allclose(a, b, rtol=2e-6, atol=1e-12)
    P = _oracle_P(kg.n_nodes, kg.edge_src, kg.edge_dst, w)
    want = ppr.ppr_batch_power(P, R.T.astype(np.float64), 0.5).T
    assert np.max(np.abs(a - want) / want.max(axis=1, keepdims=True)) < RTOL


# ------------------------------------------------------------------------------ K2: similarity
@pytest.mark.parametrize("dim,rows,bq", [(64, 1000, 5), (768, 3000, 300), (136, 777, 130), (1024, 513, 129)])
def test_similarity_modes_vs_float64(hb, dim, rows, bq):
    from hipporag_b200 import synth
    E = synth.unit_rows(rows, dim, seed=dim)
    Q = synth.unit_rows(bq, dim, seed=dim + 1)
    Q[0] = E[3]                                   # an exact match: score 1.0
    want = Q.astype(np.float64) @ E.astype(np.float64).T
    e = hb.Engine(0)
    e.load_embeddings(E, synth.unit_rows(8, dim, seed=9))
    # BF16X3: the split itself is good to ~1e-6; the rest is the tensor core's truncating fp32
    # accumulation, which biases LARGE accumulators (the planted score 1.0: ~200 accumulation steps
    # x 2^-24) -- measured 4e-6 there, 1e-7..4e-7 on ordinary scores.  Still inside the 1e-5 budget.
    for mode, tol in ((hb.SIM_FP32, 1e-6), (hb.SIM_BF16X3, 8e-6), (hb.SIM_BF16, 1.5e-2)):
        e.set_options(sim_mode=mode)
        idx_fused, score_fused, _ = e.stage_a(Q, 5)          # default: selection fused into the GEMM epilogue
        e.debug_keep_scores(True)
        idx, score, nv = e.stage_a(Q, 5)
        e.debug_keep_scores(False)
        assert np.array_equal(idx, idx_fused) and np.array_equal(score, score_fused)
        got = e.debug_scores(0)
        assert got.shape == want.shape
        assert np.max(np.abs(got - want)) < tol, (mode, np.max(np.abs(got - want)))
        if mode != hb.SIM_BF16:
            for b in range(0, bq, 17):
                assert_topk_matches(idx[b], score[b], retrieve.min_max_normalize(want[b]), 5, what=f"mode {mode} q{b}")
    assert idx[0, 0] == 3


def test_knn_matches_exact_cosine_topk(hb):
    """8(f)-2: retrieve_knn drop-in (utils/embed_utils.py:6) vs float64 cosine + deterministic top-k."""
    from hipporag_b200.knn import retrieve_knn
    rng = np.random.default_rng(0)
    keys = rng.standard_normal((3000, 64)).astype(np.float32) * rng.random((3000, 1)).astype(np.float32) * 3
    keys[10] = keys[7]                                          # exact duplicate -> tie broken by index
    qs = keys[:50] + 0.05 * rng.standard_normal((50, 64)).astype(np.float32)
    key_ids = [f"k{i}" for i in range(3000)]
    res = retrieve_knn([f"q{i}" for i in range(50)], key_ids, qs, keys, k=2047)
    kn = keys.astype(np.float64) / np.linalg.norm(keys.astype(np.float64), axis=1, keepdims=True)
    qn = qs.astype(np.float64) / np.linalg.norm(qs.astype(np.float64), axis=1, keepdims=True)
    S = qn @ kn.T
    for i in range(50):
        ids, sc = res[f"q{i}"]
        assert len(ids) == 2047 and ids[0] == ("k7" if i == 10 else f"k{i}")   # key 10 duplicates key 7
        got = np.array([int(x[1:]) for x in ids])
        sc = np.array(sc)
        assert len(set(got.tolist())) == 2047
        np.testing.assert_allclose(sc, S[i][got], atol=8e-6)               # cosine values (signed, near 0 too)
        assert np.all(np.diff(sc) <= 0)
        order = np.lexsort((np.arange(3000), -S[i]))[:2047]
        kth = S[i][order[-1]]
        for j in set(got.tolist()) ^ set(order.tolist()):
            assert abs(S[i][j] - kth) <= 2e-5
    assert res["q7"][0][:2] == ["k7", "k10"]                              # duplicate keys: lower index first


# ------------------------------------------------------------------------------ stages on C1
@pytest.fixture(scope="module")
def c1(hb, golden):
    g = golden
    r = hb.B200Retriever(int(g["n_nodes"]), g["edge_src"], g["edge_dst"], g["edge_w"], g["passage_vid"],
                         g["fact_subj_vid"], g["fact_obj_vid"], g["ent_chunk_count"], g["fact_emb"],
                         g["passage_emb"], damping=float(g["damping"]), linking_top_k=int(g["linking_top_k"]),
                         passage_node_weight=float(g["passage_node_weight"]), retrieval_top_k=int(g["topk"]))
    return r


def test_stage_a_musique1k(hb, golden, c1):
    g = golden
    c1.engine.debug_keep_scores(True)
    idx, score, nv = c1.engine.stage_a(g["q_fact"], 5)
    c1.engine.debug_keep_scores(False)
    idx2, score2, _ = c1.engine.stage_a(g["q_fact"], 5)
    assert np.array_equal(idx, idx2) and np.array_equal(score, score2)
    assert np.all(nv == 5)
    for q in range(g["q_fact"].shape[0]):
        fs = retrieve.fact_scores(g["fact_emb"], g["q_fact"][q])
        assert_topk_matches(idx[q], score[q], fs, 5, what=f"query {q} facts")
        assert list(idx[q]) == list(g["ref_fact_idx"][q])          # the reference's own run
        np.testing.assert_allclose(score[q], g["ref_fact_score"][q], atol=5e-6)
    c1.engine.debug_keep_scores(True)
    c1.engine.stage_a(g["q_fact"], 5)
    raw = c1.engine.debug_scores(0)
    c1.engine.debug_keep_scores(False)
    want = g["q_fact"].astype(np.float64) @ g["fact_emb"].astype(np.float64).T
    np.testing.assert_allclose(raw, want, atol=8e-6)


def test_retrieve_musique1k_matches_oracle(hb, golden, c1):
    g = golden
    ids, scores, fidx, fscore = c1.retrieve(g["q_fact"], g["q_pass"], topk=200)
    lu_P = g["P"]
    n_ref = 0
    for q in range(g["q_fact"].shape[0]):
        o = retrieve.retrieve_one(lu_P, g["tables"], g["fact_emb"], g["passage_emb"], g["q_fact"][q], g["q_pass"][q],
                                  top_k=None)
        full = np.empty(len(o["ids"]))
        full[o["ids"]] = o["scores"]
        assert_topk_matches(ids[q], scores[q], full, 200, what=f"query {q}")
        # and against the reference's own retrieve() where its phrase tie-break agrees with ours
        ref_seeds = set(int(v) for v in g["ref_seed_vid"][q] if v >= 0)
        if set(o["seeds"]) == ref_seeds:
            n_ref += 1
            reff = np.zeros(len(full))
            reff[g["ref_top_ids"][q]] = g["ref_top_scores"][q]
            np.testing.assert_allclose(scores[q], reff[ids[q]], rtol=RTOL, atol=0)
            # (a GPU id outside the reference's top-200 would have met a zero above) -> same top-200 SET as the
            # reference's own retrieve()
            assert set(ids[q].tolist()) == set(g["ref_top_ids"][q].tolist())
    assert n_ref >= 40


def test_resident_path_equals_host_path(hb, golden, c1):
    import torch
    g = golden
    ids, scores, _, _ = c1.retrieve(g["q_fact"], g["q_pass"], topk=200)
    dqf = torch.from_numpy(g["q_fact"]).cuda()
    dqp = torch.from_numpy(g["q_pass"]).cuda()
    oi = torch.empty((dqf.shape[0], 200), dtype=torch.int32, device="cuda")
    os_ = torch.empty((dqf.shape[0], 200), dtype=torch.float32, device="cuda")
    c1.engine.retrieve_resident(dqf, dqp, oi, os_, topk=200)
    torch.cuda.synchronize()
    assert np.array_equal(oi.cpu().numpy(), ids)
    assert np.array_equal(os_.cpu().numpy(), scores)


def test_dpr_fallback_and_filter(hb, golden, c1):
    g = golden
    Q = 6
    idx, score, nv = c1.engine.stage_a(g["q_fact"][:Q], 5)
    kept = idx.copy()
    kept[1] = -1                      # query 1: the filter kept nothing -> DPR (HippoRAG.py:467-469)
    kept[2, 2:] = -1                  # query 2: two facts kept
    flags = np.zeros(Q, dtype=np.uint8)
    flags[3] = 1                      # query 3: explicitly flagged
    ids, scores = c1.engine.stage_b(g["q_pass"][:Q], kept, score, flags, topk=50)
    for q in range(Q):
        nk = {1: 0, 2: 2}.get(q, 5)
        if q == 3:
            nk = 0
        o = retrieve.retrieve_one(g["P"], g["tables"], g["fact_emb"], g["passage_emb"], g["q_fact"][q],
                                  g["q_pass"][q], top_k=None, fact_filter=lambda c, nk=nk: c[:nk])
        assert o["mode"] == ("dpr" if nk == 0 else "ppr")
        full = np.empty(len(o["ids"]))
        full[o["ids"]] = o["scores"]
        assert_topk_matches(ids[q], scores[q], full, 50, what=f"query {q} ({o['mode']})")


def test_topk_tie_policy_and_k_larger_than_p(hb):
    # duplicate passages -> exactly equal scores: lower passage id first; k > P pads with -1
    rng = np.random.default_rng(0)
    d, P = 64, 12
    base = rng.standard_normal((4, d)).astype(np.float32)
    base /= np.linalg.norm(base, axis=1, keepdims=True)
    pemb = base[np.array([0, 1, 0, 2, 1, 0, 3, 3, 2, 1, 0, 2])]
    n_ent = 5
    n = n_ent + P
    r = hb.B200Retriever(n, [0, 1], [1, 2], [1.0, 1.0], np.arange(n_ent, n), np.zeros(0, np.int32),
                         np.zeros(0, np.int32), np.zeros(n, np.int32), np.zeros((0, d), np.float32), pemb)
    q = base[:2].copy()
    ids, scores, _, _ = r.retrieve(np.zeros((2, d), np.float32), q, topk=16)   # no facts -> DPR
    for b in range(2):
        s = retrieve.passage_scores(pemb, q[b])
        want = retrieve.order_desc(s)
        assert list(ids[b, :P]) == list(want)
        assert np.all(ids[b, P:] == -1)
        np.testing.assert_allclose(scores[b, :P], s[want], atol=2e-6)


def test_link_top_k_zero_keeps_every_phrase_and_k8(hb, golden, c1):
    """link_top_k falsy skips the phrase top-k filter (HippoRAG.py:1620); up to 8 kept facts = 16 phrases."""
    g = golden
    Q = 5
    idx, score, nv = c1.engine.stage_a(g["q_fact"][:Q], 8)
    ids, scores = c1.engine.stage_b(g["q_pass"][:Q], idx, score, None, link_top_k=0, topk=100)
    for q in range(Q):
        fs = retrieve.fact_scores(g["fact_emb"], g["q_fact"][q])
        kept = list(retrieve.top_facts(fs, 8))
        assert kept == list(idx[q])
        ps = retrieve.passage_scores(g["passage_emb"], g["q_pass"][q])
        r, phrases = retrieve.seed_vector(g["tables"], fs, kept, ps, 0, 0.05)
        assert len(phrases) > 8
        pi = ppr.ppr_power(g["P"], r, 0.5)[g["tables"].passage_vid]
        assert_topk_matches(ids[q], scores[q], pi, 100, what=f"query {q} (link_top_k=0)")


@pytest.mark.parametrize("k", [5, 10, 32])
def test_linking_top_k_is_configurable(hb, golden, c1, k):
    """config_utils.py:184: linking_top_k candidates go to the filter and up to that many facts are kept.  k <= 8 is
    selected in the GEMM epilogue, larger k by the exact radix select on the materialised scores; 40 queries take the
    mixed-precision solver with up to 64 phrase seeds per query."""
    g = golden
    Q = 40
    idx, score, nv = c1.engine.stage_a(g["q_fact"][:Q], k)
    assert np.all(nv == k)
    ids, scores = c1.engine.stage_b(g["q_pass"][:Q], idx, score, None, link_top_k=k, topk=100)
    for q in (0, 7, 19, 39):
        fs = retrieve.fact_scores(g["fact_emb"], g["q_fact"][q])
        kept = list(retrieve.top_facts(fs, k))
        assert kept == list(idx[q]), f"query {q}: top-{k} facts"
        np.testing.assert_allclose(score[q], fs[kept], atol=1e-5)
        o = retrieve.retrieve_one(g["P"], g["tables"], g["fact_emb"], g["passage_emb"], g["q_fact"][q], g["q_pass"][q],
                                  link_top_k=k, top_k=None)
        full = np.empty(len(o["ids"]))
        full[o["ids"]] = o["scores"]
        assert_topk_matches(ids[q], scores[q], full, 100, what=f"query {q} (linking_top_k={k})")


def test_error_paths_raise_instead_of_falling_back(hb, golden):
    g = golden
    e = hb.Engine(0)
    with pytest.raises((hb.HragError, ValueError)):          # tables need the graph first
        e.load_tables(g["passage_vid"], g["fact_subj_vid"], g["fact_obj_vid"], g["ent_chunk_count"])
    with pytest.raises(hb.HragError, match="graph not loaded"):
        e.bench_sweep(16, 1)
    e.load_graph(int(g["n_nodes"]), g["edge_src"], g["edge_dst"], g["edge_w"])
    with pytest.raises(hb.HragError, match="out of range"):
        e.load_tables(np.array([int(g["n_nodes"])], np.int32), g["fact_subj_vid"], g["fact_obj_vid"], g["ent_chunk_count"])
    e.load_tables(g["passage_vid"], g["fact_subj_vid"], g["fact_obj_vid"], g["ent_chunk_count"])
    with pytest.raises(hb.HragError, match="multiple of 4"):
        e.load_embeddings(np.zeros((3, 6), np.float32), np.zeros((3, 6), np.float32))
    e.load_embeddings(g["fact_emb"], g["passage_emb"])
    with pytest.raises(hb.HragError, match="must be in"):
        e.stage_a(g["q_fact"][:2], 33)
    idx, score, _ = e.stage_a(g["q_fact"][:2], 5)
    with pytest.raises(hb.HragError, match="bad sizes"):
        e.stage_b(g["q_pass"][:2], idx, score, topk=5000)
    with pytest.raises(hb.HragError, match="damping"):
        e.stage_b(g["q_pass"][:2], idx, score, damping=1.5)
    with pytest.raises(ValueError):
        e.ppr(np.ones(7, np.float32))
    # two handles on one device are independent
    e2 = hb.Engine(0)
    e2.load_graph(2, [0], [1], [1.0])
    e2.set_options(ppr_precision=hb.PPR_FP32)
    np.testing.assert_allclose(e2.ppr(np.array([1.0, 0.0])), [2 / 3, 1 / 3], atol=2e-7)
    ids, _ = e.stage_b(g["q_pass"][:2], idx, score, topk=5)
    assert ids.shape == (2, 5) and ids.min() >= 0


def test_many_queries_cross_chunk_boundaries(hb):
    """> 1024 queries: several chunks, mixed-precision sub-batches of 32 with a ragged tail; spot-check
    queries in the first chunk, across the boundary and in the tail against the oracle."""
    from hipporag_b200 import synth
    kg = synth.make_kg(5_000, 50_000, seed=21)
    d = 64
    fe, pe = synth.unit_rows(kg.n_facts, d, 3), synth.unit_rows(kg.n_pass, d, 4)
    nq = 1024 + 1024 + 77
    qf, qp, _ = synth.make_queries(kg, fe, pe, nq, seed=5)
    r = hb.B200Retriever(kg.n_nodes, kg.edge_src, kg.edge_dst, kg.edge_w, kg.passage_vid, kg.fact_subj_vid,
                         kg.fact_obj_vid, kg.ent_chunk_count, fe, pe)
    ids, scores, _, _ = r.retrieve(qf, qp, topk=100)
    P = _oracle_P(kg.n_nodes, kg.edge_src, kg.edge_dst, kg.edge_w)
    tb = retrieve.Tables(kg.n_nodes, kg.passage_vid, kg.fact_subj_vid, kg.fact_obj_vid, kg.ent_chunk_count)
    for q in (0, 31, 32, 1023, 1024, 2047, 2048, nq - 1):
        o = retrieve.retrieve_one(P, tb, fe, pe, qf[q], qp[q], top_k=None)
        full = np.empty(len(o["ids"]))
        full[o["ids"]] = o["scores"]
        assert_topk_matches(ids[q], scores[q], full, 100, what=f"query {q} of {nq}")
    ids2, scores2 = r.engine.stage_b(qp[:3], *r.engine.stage_a(qf[:3], 5)[:2], topk=500)      # topk up to 2048 (P = 500)
    assert ids2.shape == (3, 500) and sorted(ids2[0].tolist()) == list(range(500))


def test_empty_batch(hb, c1):
    idx, score, nv = c1.engine.stage_a(np.zeros((0, c1.engine.dim), np.float32), 5)
    assert idx.shape == (0, 5)
    ids, scores = c1.engine.stage_b(np.zeros((0, c1.engine.dim), np.float32), idx, score, topk=10)
    assert ids.shape == (0, 10)


# ------------------------------------------------------------------------------ synthetic C2-shaped
def test_synthetic_c2_shape_sample(hb):
    from hipporag_b200 import synth
    kg = synth.make_kg(100_000, 1_000_000, seed=0)
    d = 128
    fe = synth.unit_rows(kg.n_facts, d, seed=10)
    pe = synth.unit_rows(kg.n_pass, d, seed=11)
    qf, qp, planted = synth.make_queries(kg, fe, pe, 48, seed=12)
    r = hb.B200Retriever(kg.n_nodes, kg.edge_src, kg.edge_dst, kg.edge_w, kg.passage_vid, kg.fact_subj_vid,
                         kg.fact_obj_vid, kg.ent_chunk_count, fe, pe)
    ids, scores, fidx, fscore = r.retrieve(qf, qp, topk=200)
    assert np.array_equal(fidx[:, 0], planted)           # the planted fact is every query's best fact
    P = _oracle_P(kg.n_nodes, kg.edge_src, kg.edge_dst, kg.edge_w)
    tb = retrieve.Tables(kg.n_nodes, kg.passage_vid, kg.fact_subj_vid, kg.fact_obj_vid, kg.ent_chunk_count)
    for q in range(0, 48, 4):
        o = retrieve.retrieve_one(P, tb, fe, pe, qf[q], qp[q], top_k=None)
        full = np.empty(len(o["ids"]))
        full[o["ids"]] = o["scores"]
        assert_topk_matches(ids[q], scores[q], full, 200, what=f"C2 query {q}")
    st = r.engine.stats()
    assert st["kernel_launches"] > 0 and st["ppr_sweeps"] > 0
