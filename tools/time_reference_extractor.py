#!/usr/bin/env python
"""Time the REFERENCE'S OWN CPython extractor (src/classes.py:652-733, imported under a torch_geometric
stub by oracle/ref_import.py) and the oracle's C restatement on one host core, on the shipped NPInter2
project 1223_1 / fold 0 (SURVEY 8d: "also time the reference's own CPython extractor ... for the
extraction-only comparison").  Needs the reference tree (oracle/ref_import.py: REF_ROOT); writes profiles/ref_extractor_cpu.json.

    python tools/time_reference_extractor.py [n_pairs]
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import khop, khop_cwrap, refdata, ref_import  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
ds, keys, table = refdata.load_project(ref_import.require_reference(), "1223_1", "NPInter2", 0)
cannot = keys["set_interactionKey_test"] + keys["set_negativeInteractionKey_test"]
pool = keys["set_interactionKey_train"] + keys["set_negativeInteractionKey_train"]
rng = np.random.default_rng(20211223)
pick = [tuple(int(v) for v in pool[i]) for i in rng.choice(len(pool), size=n, replace=False)]

R = ref_import.ReferenceExtractor(ds, table, cannot)
for key in pick[:20]:
    R.extract(key)
t0 = time.perf_counter()
nodes = 0
for key in pick:
    nodes += R.extract(key).x.shape[0]
t_ref = time.perf_counter() - t0

g = khop.build_csr(ds.edges, ds.is_rna)
mask = khop.mask_from_keys(g, [tuple(k) for k in cannot])
pairs = np.asarray(pick, dtype=np.int32)
ys = np.zeros(len(pairs), dtype=np.int64)
out = {"dataset": "NPInter2 project 1223_1 fold 0 (shipped), %d train pairs, 1 core" % n,
       "reference_cpython_h1": {"subgraphs_per_s": n / t_ref, "mean_nodes": nodes / n,
                                "what": "src/classes.py:652-733 incl. its per-node feature rows (torch.tensor of Python lists)"}}
for h in (1, 2):
    khop_cwrap.collate_batch(g, mask, pairs[:50], ys[:50], h, table)
    t0 = time.perf_counter()
    for i in range(0, n, 200):
        khop_cwrap.collate_batch(g, mask, pairs[i:i + 200], ys[i:i + 200], h, table)
    out["oracle_c_h%d" % h] = {"subgraphs_per_s": n / (time.perf_counter() - t0),
                               "what": "oracle/khop_c.c extraction + collation + dense feature rows, batches of 200"}
json.dump(out, open(os.path.join(ROOT, "profiles", "ref_extractor_cpu.json"), "w"), indent=1)
print(json.dumps(out, indent=1))
