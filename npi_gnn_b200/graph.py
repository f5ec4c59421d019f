"""Device-resident bipartite interaction graph + enclosing-subgraph pair sets.

Replaces the reference's Node/LncRNA/Protein object graph (src/classes.py:19-42, built at
src/generate_edgelist.py:56-90 and extended with negatives at src/generate_dataset.py:204-216)
by a CSR in HBM, the ``set_allInteractionKey_cannotUse`` Python set (src/generate_dataset.py:297-299)
by a per-edge byte mask, and the per-node ``embedded_vector``/``attributes_vector`` lists
(src/generate_dataset.py:55-119) by one padded float32 feature table.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib as L
from . import ops


def _key64(pairs):
    pairs = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    return (pairs[:, 0] << 32) | pairs[:, 1]


class BipartiteGraph:
    """pos U neg interaction graph (negatives are structural edges, SURVEY 0.4).

    edges  : [E,2] (rna_serial, protein_serial) in the order the reference appends interactions to
             the nodes' interaction lists (xlsx rows, then rebuilt negatives).
    is_rna : [V] node type by serial number (serials interleave the two types).
    table  : [V, F-1] float32 node features WITHOUT the structural-label column
             (node2vec 64 | k-mer 113, or node2vec only for --noKmer).
    """

    def __init__(self, edges, is_rna, table, device="cuda"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.NPIError("BipartiteGraph lives in GPU memory; device must be CUDA (no CPU fallback)")
        edges = np.ascontiguousarray(edges, dtype=np.int32).reshape(-1, 2)
        is_rna = np.ascontiguousarray(is_rna, dtype=np.uint8)
        table = np.ascontiguousarray(table, dtype=np.float32)
        V = is_rna.shape[0]
        if table.shape[0] != V:
            raise L.NPIError("feature table has %d rows for %d nodes" % (table.shape[0], V))
        if len(edges) and not (is_rna[edges[:, 0]].all() and not is_rna[edges[:, 1]].any()):
            raise L.NPIError("edges must be (rna_serial, protein_serial)")
        rowptr, col, eid, edge_id, nu = ops.csr_build_host(edges, V)
        self._finish(rowptr, col, eid, edges[edge_id >= 0], is_rna, table)

    @classmethod
    def from_adjacency(cls, adjacency, is_rna, table, device="cuda"):
        """Build from per-node ordered key lists (``Node.interaction_list`` of the reference's object
        graph): adjacency[s] = [(rna_serial, protein_serial), ...].  Duplicate keys inside a list
        keep their first position; edge ids are assigned in order of first appearance."""
        self = cls.__new__(cls)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.NPIError("BipartiteGraph lives in GPU memory; device must be CUDA (no CPU fallback)")
        is_rna = np.ascontiguousarray(is_rna, dtype=np.uint8)
        table = np.ascontiguousarray(table, dtype=np.float32)
        V = len(is_rna)
        ids, rowptr, col, eid = {}, np.zeros(V + 1, dtype=np.int32), [], []
        for s in range(V):
            seen = set()
            for a, b in adjacency[s]:
                key = (int(a), int(b))
                if key in seen:
                    continue
                seen.add(key)
                if s != key[0] and s != key[1]:
                    raise L.NPIError("adjacency[%d] holds a key that does not touch node %d" % (s, s))
                eid.append(ids.setdefault(key, len(ids)))
                col.append(key[1] if key[0] == s else key[0])
            rowptr[s + 1] = len(col)
        edges = np.zeros((len(ids), 2), dtype=np.int32)
        for (a, b), e in ids.items():
            edges[e] = (a, b)
        self._finish(rowptr, np.asarray(col, dtype=np.int32), np.asarray(eid, dtype=np.int32), edges, is_rna, table)
        return self

    def _finish(self, rowptr, col, eid, edges_unique, is_rna, table):
        V = len(is_rna)
        nu = len(edges_unique)
        self.num_nodes = V
        self.num_edges = nu
        self.F = table.shape[1] + 1                      # + structural label (src/classes.py:709-712)
        self.ld = (self.F + 3) // 4 * 4
        self.edges_h = edges_unique                      # unique edges, id order
        self._keys_sorted = None
        self.rowptr_h, self.col_h, self.eid_h = rowptr, col, eid
        self.is_rna_h = is_rna
        dev = self.device
        self.rowptr = torch.from_numpy(np.ascontiguousarray(rowptr)).to(dev)
        self.col = torch.from_numpy(np.ascontiguousarray(col) if len(col) else np.zeros(1, dtype=np.int32)).to(dev)
        self.eid = torch.from_numpy(np.ascontiguousarray(eid) if len(eid) else np.zeros(1, dtype=np.int32)).to(dev)
        self.is_rna = torch.from_numpy(is_rna).to(dev)
        self.mask = torch.zeros(max(nu, 1), dtype=torch.uint8, device=dev)
        self.mask_h = np.zeros(max(nu, 1), dtype=np.uint8)
        self.max_degree = int(np.diff(rowptr).max()) if V else 0
        self.colm = torch.empty_like(self.col)           # col with the edge mask folded into bit 31
        self._fold_mask()
        padded = np.zeros((V, self.ld), dtype=np.float32)   # column 0 is reserved for the label
        padded[:, 1:self.F] = table
        self.table = torch.from_numpy(padded).to(dev)
        self.table_h = table

    # -- edge ids / mask --------------------------------------------------------------------
    def edge_ids(self, pairs):
        """Undirected edge id of every (rna, protein) key, -1 if the key is not an edge."""
        if self._keys_sorted is None:
            k = _key64(self.edges_h)
            order = np.argsort(k, kind="stable")
            self._keys_sorted = (k[order], order.astype(np.int32))
        ks, order = self._keys_sorted
        q = _key64(pairs)
        pos = np.searchsorted(ks, q)
        pos = np.clip(pos, 0, max(len(ks) - 1, 0))
        hit = (ks[pos] == q) if len(ks) else np.zeros(len(q), dtype=bool)
        return np.where(hit, order[pos], -1).astype(np.int32)

    def candidate_pairs(self):
        """Every (rna, protein) pair that is not an edge, RNA-major in serial order: int32 [R * P - E, 2].  Negatives are
        edges too (SURVEY 0.4), so these are the pairs that are neither a known interaction nor a sampled negative --
        the list a case study scores.  Host only."""
        r = np.nonzero(self.is_rna_h)[0].astype(np.int32)
        p = np.nonzero(self.is_rna_h == 0)[0].astype(np.int32)
        allp = np.stack([np.repeat(r, len(p)), np.tile(p, len(r))], 1)
        return allp[self.edge_ids(allp) < 0]

    def _fold_mask(self):
        if len(self.col_h):
            ops.csr_fold_mask(self.col, self.eid, self.mask, self.colm)
        else:
            self.colm.copy_(self.col)

    def set_mask(self, cannot_use_pairs):
        """``set_allInteractionKey_cannotUse``: keys hidden from expansion (the target edge of a
        pair is exempt, src/classes.py:668)."""
        m = np.zeros(max(self.num_edges, 1), dtype=np.uint8)
        if cannot_use_pairs is not None and len(cannot_use_pairs):
            ids = self.edge_ids(cannot_use_pairs)
            m[ids[ids >= 0]] = 1
        self.mask_h = m
        self.mask.copy_(torch.from_numpy(m))
        self._fold_mask()
        return self

    def features_for(self, gid, dist):
        return L.features_virtual(self.table, gid, dist, self.F)


def _khop_ctas(V, budget_bytes=2 << 30):
    sms = ops.sm_count()
    per = ops.khop_workspace_bytes(V, 1)
    return int(max(1, min(2 * sms, budget_bytes // max(per, 1))))


class PairSet:
    """A resident set of target pairs with labels and cached per-pair subgraph sizes.

    Equivalent of one ``LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory`` instance
    (src/classes.py:602-650): the list of interactions to generate subgraphs for, with h hops.
    The count pass of the GPU extractor runs once here (like ``process()`` runs once); subgraphs
    themselves are re-extracted on the GPU whenever a batch is assembled."""

    def __init__(self, graph: BipartiteGraph, pairs, y, h=1):
        self.graph = graph
        self.h = int(h)
        dev = graph.device
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        y = np.ascontiguousarray(y, dtype=np.int32).reshape(-1)
        if len(pairs) != len(y):
            raise L.NPIError("pairs and y differ in length")
        if len(pairs):
            V = graph.num_nodes
            if pairs.min() < 0 or pairs.max() >= V:
                raise L.NPIError("pair serial out of range")
            if not (graph.is_rna_h[pairs[:, 0]].all() and not graph.is_rna_h[pairs[:, 1]].any()):
                raise L.NPIError("pairs must be (rna_serial, protein_serial)")
        self.pairs_h, self.y_h = pairs, y
        P = len(pairs)
        self.pairs = torch.from_numpy(pairs).to(dev)
        self.y = torch.from_numpy(y).to(dev)
        self.n_all = torch.zeros(max(P, 1), dtype=torch.int32, device=dev)
        self.e_all = torch.zeros(max(P, 1), dtype=torch.int32, device=dev)
        self.num_ctas = _khop_ctas(graph.num_nodes)
        self.khop_ws = torch.empty(ops.khop_workspace_bytes(graph.num_nodes, self.num_ctas), dtype=torch.uint8, device=dev)
        if P:
            ops.khop_count(graph, self.pairs, self.h, self.n_all, self.e_all, self.khop_ws, self.num_ctas)
        self.n_h = self.n_all.cpu().numpy()[:P].astype(np.int64)
        self.e_h = self.e_all.cpu().numpy()[:P].astype(np.int64)
        self.max_nodes = int(self.n_h.max()) if P else 2     # node capacity of the fill pass

    def __len__(self):
        return len(self.pairs_h)

    def batch_caps(self, batch_size, order=None):
        """Largest (N0, E0, n_graph) over the batches of a sequential pass in ``order`` (pair indices, any length;
        default: the whole pair set)."""
        idx = np.arange(len(self)) if order is None else np.asarray(order)
        n, e = self.n_h[idx], self.e_h[idx]
        starts = np.arange(0, len(idx), batch_size)
        return int(np.add.reduceat(n, starts).max()), int(np.add.reduceat(e, starts).max()), int(n.max())
