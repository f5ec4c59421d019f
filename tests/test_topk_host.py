"""Host side of the per-node ranking: BipartiteGraph.candidate_pairs and the argument check of top_k_by_group (no GPU)."""
import numpy as np
import pytest

from tests.common import synthetic_bipartite


def _host_graph(d):
    """A BipartiteGraph with its host fields only: candidate_pairs and edge_ids read nothing else."""
    from npi_gnn_b200.graph import BipartiteGraph
    g = BipartiteGraph.__new__(BipartiteGraph)
    g.edges_h, g.is_rna_h, g._keys_sorted = d["edges"], d["is_rna"], None
    return g


@pytest.mark.parametrize("seed", [11, 12])
def test_candidate_pairs_are_every_non_edge(seed):
    d = synthetic_bipartite(seed, 60, 40, 300, 300)
    cand = _host_graph(d).candidate_pairs()
    is_rna = d["is_rna"].astype(bool)
    want = {(int(r), int(p)) for r in np.nonzero(is_rna)[0] for p in np.nonzero(~is_rna)[0]} \
        - {tuple(e) for e in d["edges"].tolist()}
    assert cand.dtype == np.int32 and cand.shape == (len(want), 2)
    assert {tuple(c) for c in cand.tolist()} == want
    assert (_host_graph(d).edge_ids(cand) < 0).all()
    key = cand[:, 0].astype(np.int64) * len(is_rna) + cand[:, 1]
    assert (np.diff(key) > 0).all()                                 # RNA-major, serial order


def test_top_k_by_group_rejects_k_before_touching_the_device():
    import torch
    from npi_gnn_b200 import top_k_by_group
    for k in (0, 1025):
        with pytest.raises(ValueError):
            top_k_by_group(torch.zeros(4), torch.zeros(4, dtype=torch.int32), 1, k)
