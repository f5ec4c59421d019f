"""Run the REFERENCE's own extractor (src/classes.py:652-733) in this container.

Needs a checkout of the reference (REF_ROOT below): it registers a minimal ``torch_geometric``
stub so that ``src/classes.py`` imports unchanged (its imports are at src/classes.py:1-5),
rebuilds the reference's object graph from a RawDataset exactly as
src/generate_edgelist.py:61-98 and src/generate_dataset.py:204-216 do, and calls
``LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory.local_subgraph_generation`` as an
unbound function.  Used by tools/make_golden.py and by tests that are skipped when the
reference tree is absent (e.g. on the GPU box).  Nothing here is copied from the reference;
the reference module is imported from where it lies.
"""
from __future__ import annotations

import os
import sys
import types

# a checkout of the reference: $NPI_REFERENCE_ROOT, else oracle/_ref (git-ignored, never committed).  The tests that
# read it are skipped when it is absent (marker `reference`); the tools that read it stop in require_reference().
REF_ROOT = os.environ.get("NPI_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def reference_available():
    return os.path.exists(os.path.join(REF_ROOT, "src", "classes.py"))


def require_reference():
    """REF_ROOT, or one clear error when no reference tree is there."""
    if not reference_available():
        raise SystemExit("no reference tree at %s: put a checkout of AshuiRUA/NPI-GNN there or set NPI_REFERENCE_ROOT"
                         % REF_ROOT)
    return REF_ROOT


def _install_stub():
    if "torch_geometric" in sys.modules and getattr(sys.modules["torch_geometric"], "_npi_stub", False):
        return
    import torch

    tg = types.ModuleType("torch_geometric")
    tg._npi_stub = True
    tgnn = types.ModuleType("torch_geometric.nn")
    tgdata = types.ModuleType("torch_geometric.data")

    class _Empty(torch.nn.Module):
        def __init__(self, *a, **k):
            super().__init__()

    for nm in ("GCNConv", "TopKPooling", "SAGEConv", "EdgePooling"):
        setattr(tgnn, nm, type(nm, (_Empty,), {}))
    tgnn.global_mean_pool = lambda *a, **k: None
    tgnn.global_max_pool = lambda *a, **k: None

    class Data:
        def __init__(self, x=None, y=None, edge_index=None):
            self.x, self.y, self.edge_index = x, y, edge_index

    class Dataset:
        pass

    class InMemoryDataset:
        pass

    tgdata.Data, tgdata.Dataset, tgdata.InMemoryDataset = Data, Dataset, InMemoryDataset
    tg.nn, tg.data = tgnn, tgdata
    sys.modules["torch_geometric"] = tg
    sys.modules["torch_geometric.nn"] = tgnn
    sys.modules["torch_geometric.data"] = tgdata


def import_reference_classes():
    require_reference()
    _install_stub()
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import importlib
    return importlib.import_module("src.classes")


class ReferenceExtractor:
    """The reference's object graph + its live 1-hop extractor."""

    def __init__(self, raw, table, cannot_use):
        """raw: oracle.refdata.RawDataset (negatives already rebuilt); table: [V,F-1] float32
        (emb | k-mer); cannot_use: iterable of (rna_serial, prot_serial) keys."""
        C = import_reference_classes()
        self.C = C
        self.nodes = []
        for s, nm in enumerate(raw.names):
            node = (C.LncRNA(nm, s, "LncRNA") if raw.is_rna[s] else C.Protein(nm, s, "Protein"))
            # read_node2vec_result leaves the embedding as strings and classes.py:713 calls float();
            # repr(float32->float) round-trips to the same float32, which is all that reaches x.
            node.embedded_vector = [repr(float(v)) for v in table[s, :64]]
            node.attributes_vector = [float(v) for v in table[s, 64:]]
            self.nodes.append(node)
        self.interactions = {}
        pos = set(raw.pos)
        # interaction_list order per node == raw.adj order (xlsx rows, then rebuilt negatives)
        made = {}
        for s in range(raw.num_nodes):
            for key in raw.adj[s]:
                it = made.get(key)
                if it is None:
                    it = C.LncRNA_Protein_Interaction(self.nodes[key[0]], self.nodes[key[1]],
                                                      1 if key in pos else 0, key)
                    made[key] = it
                self.nodes[s].interaction_list.append(it)
        self.interactions = made
        self._self = types.SimpleNamespace(sum_node=0.0, set_allInteractionKey_cannotUse=set(cannot_use))
        self._fn = C.LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory.local_subgraph_generation

    def extract(self, key, y=None):
        """Returns the reference's Data(x, y, edge_index) for the pair ``key``.  A pair that is
        not an edge of the graph (candidate scoring) gets a fresh interaction object, like
        src/case_study_negativeSample.py:339-349 does for test negatives."""
        it = self.interactions.get(key)
        if it is None:
            it = self.C.LncRNA_Protein_Interaction(self.nodes[key[0]], self.nodes[key[1]], 0 if y is None else y, key)
        return self._fn(self._self, it, 1)
