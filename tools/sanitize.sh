#!/bin/bash
# compute-sanitizer passes over a small end-to-end run of every kernel family (SURVEY.md 5: race detection).
# Usage (GPU box): bash tools/sanitize.sh [memcheck|racecheck|synccheck|initcheck]
set -u
TOOL=${1:-memcheck}
cat > /tmp/hrag_sanitize_driver.py <<'PY'
import numpy as np, sys, os
sys.path.insert(0, os.getcwd())
import hipporag_b200 as hb
from hipporag_b200 import synth
kg = synth.make_kg(3000, 30000, seed=5)
d = 64
fe, pe = synth.unit_rows(kg.n_facts, d, 1), synth.unit_rows(kg.n_pass, d, 2)
qf, qp, _ = synth.make_queries(kg, fe, pe, 40, seed=3)
# a hub row > 256 nnz so the long-row kernels run too
src = np.concatenate([kg.edge_src, np.zeros(400, np.int32)]); dst = np.concatenate([kg.edge_dst, np.arange(1, 401, dtype=np.int32)])
w = np.concatenate([kg.edge_w, np.ones(400)])
r = hb.B200Retriever(kg.n_nodes, src, dst, w, kg.passage_vid, kg.fact_subj_vid, kg.fact_obj_vid, kg.ent_chunk_count, fe, pe)
for prec in (hb.PPR_MIXED, hb.PPR_FP32):
    for sim in (hb.SIM_BF16X3, hb.SIM_BF16, hb.SIM_FP32):
        r.engine.set_options(ppr_precision=prec, sim_mode=sim)
        ids, sc, _, _ = r.retrieve(qf, qp, topk=50)
        ids2, sc2, _, _ = r.retrieve(qf[:5], qp[:5], topk=50)
r.engine.set_options(ppr_precision=hb.PPR_MIXED, sim_mode=hb.SIM_BF16X3)
R = np.random.default_rng(0).random((3, kg.n_nodes), dtype=np.float32)
r.engine.ppr(R)
r.engine.ppr(np.random.default_rng(1).random((20, kg.n_nodes), dtype=np.float32), damping=0.85)
r.engine.similarity(1, qp[:3])
# round-2 kernels: linking_top_k > 8 (radix select path + 64 seed slots), threshold KNN epilogue
idx, score, nv = r.engine.stage_a(qf, 10)
r.engine.stage_b(qp, idx, score, link_top_k=10, topk=50)
r.engine.knn_threshold(0, fe[:200], 0.3, 64)
print("driver ok", ids.shape)
PY
compute-sanitizer --tool $TOOL --error-exitcode 7 python /tmp/hrag_sanitize_driver.py 2>&1 | tail -15
echo "sanitizer($TOOL) exit: $?"
