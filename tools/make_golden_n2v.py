#!/usr/bin/env python
"""Golden vectors for the node2vec stage from the REFERENCE'S OWN code (needs the reference tree, oracle/ref_import.py):
imports <reference>/node2vec-master/src/node2vec.py (the only patch: `np.int = int`, an alias
numpy >= 1.24 removed), builds the graph like main.py:read_graph (:63-76) and stores the alias tables
(J, q) of preprocess_transition_probs for
  * a small NON-bipartite graph with triangles (all three branches of get_alias_edge), p = 0.5, q = 2,
  * a small bipartite graph, p = 1, q = 1 (the reference's defaults, main.py:48-52),
  * the real NPInter2 fold-0 training graph (src/generate_edgelist.py:497-508: whole graph minus the test
    keys): every node table and the edge tables of 300 sampled directed edges incl. the largest hub, p = 0.25, q = 4.
Output: tests/golden/n2v_alias.npz.   Usage: python tools/make_golden_n2v.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import                            # noqa: E402
np.int = int                                             # noqa: removed alias the reference still uses (node2vec.py:114)
sys.path.insert(0, os.path.join(ref_import.require_reference(), "node2vec-master", "src"))
import networkx as nx                                    # noqa: E402
import node2vec as ref                                   # noqa: E402


def ref_graph(edges):
    G = nx.DiGraph()
    for a, b in edges:
        G.add_edge(int(a), int(b))
    for e in G.edges():
        G[e[0]][e[1]]["weight"] = 1
    return G.to_undirected()


def tables(edges, p, q, edge_sample=None):
    G = ref_graph(edges)
    g = ref.Graph(G, False, p, q)
    nodes = sorted(G.nodes())
    nJ, nq, nptr = [], [], [0]
    for v in nodes:
        un = [G[v][n]["weight"] for n in sorted(G.neighbors(v))]
        norm = sum(un)
        J, qq = ref.alias_setup([float(u) / norm for u in un])
        nJ.append(J); nq.append(qq); nptr.append(nptr[-1] + len(J))
    if edge_sample is None:
        pairs = [(s, d) for s in nodes for d in sorted(G.neighbors(s))]
    else:
        pairs = edge_sample
    eJ, eq, eptr = [], [], [0]
    for s, d in pairs:
        J, qq = g.get_alias_edge(s, d)
        eJ.append(J); eq.append(qq); eptr.append(eptr[-1] + len(J))
    return dict(nodes=np.asarray(nodes, dtype=np.int32), node_ptr=np.asarray(nptr, dtype=np.int64),
                node_J=np.concatenate(nJ).astype(np.int32), node_q=np.concatenate(nq),
                pairs=np.asarray(pairs, dtype=np.int32), edge_ptr=np.asarray(eptr, dtype=np.int64),
                edge_J=np.concatenate(eJ).astype(np.int32), edge_q=np.concatenate(eq))


def main():
    out = {}
    rng = np.random.default_rng(11)
    # (a) small general graph with triangles
    ea = set()
    while len(ea) < 60:
        a, b = rng.integers(0, 24, size=2)
        if a != b:
            ea.add((min(a, b), max(a, b)))
    ea = np.asarray(sorted(ea), dtype=np.int32)
    out["a_edges"] = ea
    for k, v in tables(ea.tolist(), 0.5, 2.0).items():
        out["a_" + k] = v
    # (b) small bipartite graph, default p = q = 1
    eb = set()
    while len(eb) < 50:
        eb.add((int(rng.integers(0, 12)), 12 + int(rng.integers(0, 9))))
    eb = np.asarray(sorted(eb), dtype=np.int32)
    out["b_edges"] = eb
    for k, v in tables(eb.tolist(), 1.0, 1.0).items():
        out["b_" + k] = v
    # (c) real NPInter2 fold-0 training graph
    z = np.load(os.path.join(ROOT, "tests", "golden", "npinter2_fold0.npz"))
    test = set(map(tuple, np.concatenate([z["test_pos"], z["test_neg"]]).tolist()))
    ec = np.asarray([e for e in z["edges"].tolist() if tuple(e) not in test], dtype=np.int32)
    G = ref_graph(ec.tolist())
    deg = dict(G.degree())
    hub = max(deg, key=deg.get)
    nodes = sorted(G.nodes())
    pick = [(hub, sorted(G.neighbors(hub))[0]), (sorted(G.neighbors(hub))[3], hub)]
    allp = [(s, d) for s in nodes for d in sorted(G.neighbors(s))]
    for i in rng.choice(len(allp), 298, replace=False):
        pick.append(allp[int(i)])
    out["c_num_train_edges"] = np.int64(len(ec))
    for k, v in tables(ec.tolist(), 0.25, 4.0, edge_sample=pick).items():
        out["c_" + k] = v
    path = os.path.join(ROOT, "tests", "golden", "n2v_alias.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, {k: v.shape for k, v in out.items() if hasattr(v, "shape")}, os.path.getsize(path))


if __name__ == "__main__":
    main()
