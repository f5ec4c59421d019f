#!/usr/bin/env python
"""Times the REFERENCE'S OWN node2vec stage (needs the reference tree, oracle/ref_import.py; imports
<reference>/node2vec-master/src/node2vec.py with the one patch `np.int = int`) on the real NPInter2
fold-0 training graph with main.py's defaults (p = q = 1, walk length 80): preprocess_transition_probs
(all alias tables) and ONE pass of simulate_walks (the reference runs ten).  gensim is absent from this
image, so Word2Vec itself cannot be timed.  Writes profiles/ref_node2vec_cpu.json."""
import contextlib
import io
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import                            # noqa: E402
np.int = int                                             # noqa
sys.path.insert(0, os.path.join(ref_import.require_reference(), "node2vec-master", "src"))
import networkx as nx                                    # noqa: E402
import node2vec as ref                                   # noqa: E402

z = np.load(os.path.join(ROOT, "tests", "golden", "npinter2_fold0.npz"))
test = set(map(tuple, np.concatenate([z["test_pos"], z["test_neg"]]).tolist()))
G = nx.DiGraph()
for a, b in z["edges"].tolist():
    if (a, b) not in test:
        G.add_edge(a, b)
for e in G.edges():
    G[e[0]][e[1]]["weight"] = 1
G = G.to_undirected()
g = ref.Graph(G, False, 1, 1)
t0 = time.perf_counter()
g.preprocess_transition_probs()
t1 = time.perf_counter()
with contextlib.redirect_stdout(io.StringIO()):
    walks = g.simulate_walks(1, 80)
t2 = time.perf_counter()
slots = sum(len(v[0]) for v in g.alias_edges.values())
out = dict(graph="NPInter2 1223_1 fold-0 training graph", nodes=G.number_of_nodes(), edges=G.number_of_edges(),
           second_order_slots=slots, preprocess_transition_probs_s=t1 - t0, simulate_walks_one_pass_s=t2 - t1,
           walks=len(walks), walks_per_s=len(walks) / (t2 - t1), ten_passes_estimate_s=10 * (t2 - t1),
           cores=1, python=sys.version.split()[0], note="reference code, CPython, one core; Word2Vec (gensim) not installed here")
json.dump(out, open(os.path.join(ROOT, "profiles", "ref_node2vec_cpu.json"), "w"), indent=1)
print(json.dumps(out))
