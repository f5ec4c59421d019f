"""Host side of the node2vec stage (no GPU): file formats, the per-fold training graph, the sorted CSR the
kernels walk, vocabulary statistics and the command-line flags -- against the oracle and, where the
reference tree is present (build container), against the reference's own source and shipped files."""
import os
import re

import numpy as np
import pytest

from npi_gnn_b200 import node2vec as n2v
from oracle import node2vec as on2v, ref_import
from tests.common import GOLD

REF = ref_import.REF_ROOT


def test_edgelist_round_trip_and_training_graph(tmp_path):
    z = np.load(os.path.join(GOLD, "npinter2_fold0.npz"))
    gold = np.load(os.path.join(GOLD, "n2v_alias.npz"))
    test_keys = np.concatenate([z["test_pos"], z["test_neg"]])
    tr = n2v.training_graph_edges(z["edges"], test_keys)
    assert len(tr) == int(gold["c_num_train_edges"]) == len(z["edges"]) - len(test_keys)
    p = str(tmp_path / "g" / "bipartite_graph.edgelist")
    n2v.write_edgelist(p, tr)
    first = open(p).readline()
    assert re.fullmatch(r"\d+ \d+ \{\}\n", first)                         # networkx' "a b {}" (what the reference writes)
    assert np.array_equal(n2v.read_edgelist(p), tr)
    # reversed test keys remove the same undirected edges
    assert len(n2v.training_graph_edges(z["edges"], test_keys[:, ::-1])) == len(tr)


def test_sorted_csr_equals_the_oracle_graph():
    gold = np.load(os.path.join(GOLD, "n2v_alias.npz"))
    for case in ("a", "b"):
        V, rowptr, col, w, nodes = n2v._sorted_csr(gold[case + "_edges"], None, False, None)
        g = on2v.SortedGraph(gold[case + "_edges"])
        assert V == g.V and np.array_equal(rowptr, g.rowptr) and np.array_equal(col, g.col)
        assert nodes.tolist() == g.nodes() == gold[case + "_nodes"].tolist()
    # duplicates and both orientations collapse; directed keeps one direction and counts sinks as nodes
    V, rowptr, col, w, nodes = n2v._sorted_csr([(0, 1), (1, 0), (0, 1), (2, 1)], None, False, None)
    assert rowptr.tolist() == [0, 1, 3, 4] and col.tolist() == [1, 0, 2, 1]
    V, rowptr, col, w, nodes = n2v._sorted_csr([(0, 3), (0, 1)], [2.0, 5.0], True, None)
    assert rowptr.tolist() == [0, 2, 2, 2, 2] and col.tolist() == [1, 3] and w.tolist() == [5.0, 2.0] and nodes.tolist() == [0, 1, 3]
    gd = on2v.SortedGraph([(0, 3), (0, 1)], directed=True)
    assert gd.nodes() == nodes.tolist()


def test_vocab_statistics_equal_the_oracle():
    rng = np.random.default_rng(2)
    walks = [rng.integers(0, 30, size=rng.integers(2, 40)).tolist() for _ in range(60)]
    cnt, keep, pneg = on2v.sg_vocab(walks, 32)
    k2, p2 = n2v.vocab_statistics(cnt)
    assert np.array_equal(k2, keep) and np.array_equal(p2, pneg)
    assert k2[30] == 0.0 and p2[31] == 0.0 and abs(p2.sum() - 1) < 1e-12


def test_word2vec_text_format(tmp_path):
    rng = np.random.default_rng(3)
    vec = rng.standard_normal((5, 64)).astype(np.float32)
    nodes = [7, 2, 9, 0, 4]
    p = str(tmp_path / "r" / "result.emb")
    n2v.save_word2vec_format(p, nodes, vec)
    lines = open(p).read().splitlines()
    assert lines[0] == "5 64" and len(lines) == 6 and lines[1].split()[0] == "7" and len(lines[1].split()) == 65
    emb = n2v.load_word2vec_format(p, 12)
    assert np.allclose(emb[nodes], vec, rtol=1e-6) and not emb[[1, 3, 5, 6, 8, 10, 11]].any()


@pytest.mark.reference
def test_flags_and_files_against_the_live_reference():
    src = open(os.path.join(REF, "node2vec-master/src/main.py")).read()
    ref_flags = {}
    for m in re.finditer(r"add_argument\('(--[\w-]+)'[^)]*?default=([^,\n)]+)", src):
        ref_flags[m.group(1)] = m.group(2).strip()
    a = n2v.parse_args([])
    for flag, default in ref_flags.items():
        name = flag[2:].replace("-", "_")
        if name in ("input", "output"):
            continue
        assert str(getattr(a, name)) == default.strip("'\""), flag
    assert a.weighted is False and a.directed is False
    # the shipped result.emb parses with our reader exactly like oracle/refdata.py's
    from oracle import refdata
    path = os.path.join(REF, "data/node2vec_result/1223_1/training_0/result.emb")
    emb = n2v.load_word2vec_format(path, 5085)
    assert np.array_equal(emb, refdata.read_node2vec(path, 5085))
    assert np.count_nonzero(np.abs(emb).sum(1)) == 4976
    # and the shipped edgelist of the fold equals our generate_G_training
    z = np.load(os.path.join(GOLD, "npinter2_fold0.npz"))
    ours = n2v.training_graph_edges(z["edges"], np.concatenate([z["test_pos"], z["test_neg"]]))
    shipped = n2v.read_edgelist(os.path.join(REF, "data/graph/1223_1/training_0/bipartite_graph.edgelist"))
    canon = lambda e: set(map(tuple, np.sort(e, axis=1).tolist()))      # noqa: E731
    assert canon(ours) == canon(shipped)
