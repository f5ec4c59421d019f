#!/usr/bin/env python
"""Generate tests/golden/ from the reference tree (run in the build container only).

  python tools/make_golden.py            # needs the reference tree (oracle/ref_import.py: REF_ROOT)

What is produced and where it comes from
  npinter2_fold0.npz   the reference's shipped NPInter2 inputs for project 1223_1 / fold 0 in
                       array form (ordered edge list, node types, feature table, fold key
                       sets) -- read with oracle/refdata.py from data/source_database_data/
                       NPInter2.xlsx, data/set_allInteractionKey/1223_1/*, data/node2vec_result/
                       1223_1/training_0/result.emb, data/lncRNA_3_mer, data/protein_2_mer.
  ckpt_*.npz           seven shipped state dicts (result/1223_1/model_0_fold/{5,15,30,50},
                       result/1223_1_noKmer/model_0_fold/{20,35,50}) as plain arrays.
  kat.json             the known answers: confusion matrices implied by the metric lines of
                       result/1223_1/log_0.txt and result/1223_1_noKmer/log_0.txt, and the
                       case-study partitions data/case_study/1223_1_fold_0_negativeSamples*/
                       logs/case_predict_positive.txt mapped to (rna, protein) serial pairs.
  ref_extract_h1.npz   outputs of the REFERENCE'S OWN local_subgraph_generation
                       (src/classes.py:652-733, imported under a torch_geometric stub by
                       oracle/ref_import.py) for a fixed sample of pairs: node count, sha256 of
                       x, and the sorted directed edge list.
  toy_*.npz            tiny hand-checkable graphs run through the same reference function.
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import refdata, khop, ref_import  # noqa: E402

REF = ref_import.require_reference()
OUT = os.path.join(ROOT, "tests", "golden")


parse_log = refdata.parse_metric_log


def main():
    os.makedirs(OUT, exist_ok=True)
    ds, keys, table = refdata.load_project(REF, "1223_1", "NPInter2", 0)
    edges = np.asarray(ds.edges, dtype=np.int32)
    np.savez_compressed(
        os.path.join(OUT, "npinter2_fold0.npz"),
        edges=edges, is_rna=np.asarray(ds.is_rna, dtype=np.uint8), table=table,
        num_pos=np.int64(len(ds.pos)),
        train_pos=np.asarray(keys["set_interactionKey_train"], dtype=np.int32),
        train_neg=np.asarray(keys["set_negativeInteractionKey_train"], dtype=np.int32),
        test_pos=np.asarray(keys["set_interactionKey_test"], dtype=np.int32),
        test_neg=np.asarray(keys["set_negativeInteractionKey_test"], dtype=np.int32))

    for proj, eps in (("1223_1", (5, 15, 30, 50)), ("1223_1_noKmer", (20, 35, 50))):
        for ep in eps:
            sd = torch.load(os.path.join(REF, "result", proj, "model_0_fold", str(ep)), map_location="cpu")
            np.savez_compressed(os.path.join(OUT, "ckpt_%s_%d.npz" % (proj, ep)),
                                **{k: v.numpy() for k, v in sd.items()})

    kat = {"confusion": {}, "case_study": {}}
    npos, nneg = len(keys["set_interactionKey_test"]), len(keys["set_negativeInteractionKey_test"])
    for proj in ("1223_1", "1223_1_noKmer"):
        kat["confusion"][proj] = parse_log(os.path.join(REF, "result", proj, "log_0.txt"), npos, nneg)
    serial = {}
    for s, nm in enumerate(ds.names):
        serial[(nm, bool(ds.is_rna[s]))] = s
    for tag, d in (("0.5", "1223_1_fold_0_negativeSamples"), ("0.95", "1223_1_fold_0_negativeSamples_threshold_0.95")):
        pairs = []
        for line in open(os.path.join(REF, "data", "case_study", d, "logs", "case_predict_positive.txt")):
            a = line.rstrip("\n").split("\t")
            if len(a) < 2:
                continue
            pairs.append([serial[(a[0], True)], serial[(a[1], False)]])
        kat["case_study"][tag] = dict(ckpt="ckpt_1223_1_15.npz", positives=sorted(pairs))
    json.dump(kat, open(os.path.join(OUT, "kat.json"), "w"), indent=1, sort_keys=True)

    # ---- the reference's own extractor on a fixed sample ---------------------------------
    cannot = keys["set_interactionKey_test"] + keys["set_negativeInteractionKey_test"]
    R = ref_import.ReferenceExtractor(ds, table, cannot)
    rng = np.random.default_rng(20211223)
    pool = (keys["set_interactionKey_train"] + keys["set_negativeInteractionKey_train"]
            + keys["set_interactionKey_test"] + keys["set_negativeInteractionKey_test"])
    pick = rng.choice(len(pool), size=96, replace=False)
    # plus the biggest hubs and a never-seen candidate pair
    g = khop.build_csr(ds.edges, ds.is_rna)
    deg = np.diff(g.rowptr)
    hub_p = int(np.argmax(np.where(np.asarray(ds.is_rna) == 0, deg, -1)))
    hub_r = int(np.argmax(np.where(np.asarray(ds.is_rna) == 1, deg, -1)))
    sample = [pool[i] for i in pick] + [(hub_r, hub_p)]
    allkeys = set(ds.edges)
    cand = next((a, b) for a in ds.rna_serials() for b in ds.protein_serials() if (a, b) not in allkeys)
    sample.append(cand)
    ns, shas, eptr, eflat = [], [], [0], []
    for key in sample:
        d = R.extract(tuple(int(v) for v in key))
        x = d.x.numpy()
        ns.append(x.shape[0])
        shas.append(hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest())
        e = sorted(map(tuple, d.edge_index.numpy().T.tolist()))
        eflat.extend(e)
        eptr.append(len(eflat))
    np.savez_compressed(os.path.join(OUT, "ref_extract_h1.npz"),
                        pairs=np.asarray(sample, dtype=np.int32), n=np.asarray(ns, dtype=np.int32),
                        x_sha256=np.asarray(shas), edge_ptr=np.asarray(eptr, dtype=np.int64),
                        edges_sorted=np.asarray(eflat, dtype=np.int32))

    # ---- toy graph through the reference function ----------------------------------------
    toy = refdata.RawDataset()
    #  RNAs a0,a1,a2 ; proteins b0,b1,b2 ; serials interleaved by first appearance
    rows = [("a0", "b0"), ("a0", "b1"), ("a1", "b0"), ("a2", "b1"), ("a1", "b2"), ("a2", "b2"), ("a0", "b2")]
    rs, ps = {}, {}
    for a, b in rows:
        for nm, dct, isr in ((a, rs, True), (b, ps, False)):
            if nm not in dct:
                dct[nm] = len(toy.names); toy.names.append(nm); toy.is_rna.append(isr); toy.adj.append([])
        key = (rs[a], ps[b])
        toy.adj[key[0]].append(key); toy.adj[key[1]].append(key); toy.edges.append(key); toy.pos.append(key)
    ttab = np.random.default_rng(1).standard_normal((len(toy.names), 5)).astype(np.float32)
    # the reference hard-codes nothing about widths inside local_subgraph_generation
    Rt = ref_import.ReferenceExtractor.__new__(ref_import.ReferenceExtractor)
    cannot_t = [toy.edges[2]]
    C = ref_import.import_reference_classes()
    Rt.C = C
    Rt.nodes = []
    for s, nm in enumerate(toy.names):
        node = C.LncRNA(nm, s, "LncRNA") if toy.is_rna[s] else C.Protein(nm, s, "Protein")
        node.embedded_vector = [repr(float(v)) for v in ttab[s, :2]]
        node.attributes_vector = [float(v) for v in ttab[s, 2:]]
        Rt.nodes.append(node)
    made = {}
    for s in range(len(toy.names)):
        for key in toy.adj[s]:
            it = made.setdefault(key, C.LncRNA_Protein_Interaction(Rt.nodes[key[0]], Rt.nodes[key[1]], 1, key))
            Rt.nodes[s].interaction_list.append(it)
    Rt.interactions = made
    import types
    Rt._self = types.SimpleNamespace(sum_node=0.0, set_allInteractionKey_cannotUse=set(cannot_t))
    Rt._fn = C.LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory.local_subgraph_generation
    tx, te, tn = [], [], []
    tpairs = list(toy.edges) + [(rs["a1"], ps["b1"])]
    for key in tpairs:
        d = Rt.extract(key)
        tx.append(d.x.numpy()); tn.append(d.x.shape[0])
        te.append(np.asarray(sorted(map(tuple, d.edge_index.numpy().T.tolist())), dtype=np.int32))
    np.savez_compressed(os.path.join(OUT, "toy_h1.npz"), edges=np.asarray(toy.edges, dtype=np.int32),
                        is_rna=np.asarray(toy.is_rna, dtype=np.uint8), table=ttab,
                        masked_edge=np.asarray(cannot_t, dtype=np.int32),
                        pairs=np.asarray(tpairs, dtype=np.int32), n=np.asarray(tn, dtype=np.int32),
                        x=np.concatenate(tx), e_ptr=np.cumsum([0] + [len(e) for e in te]),
                        edges_sorted=np.concatenate(te))
    for f in sorted(os.listdir(OUT)):
        print("%10d  %s" % (os.path.getsize(os.path.join(OUT, f)), f))


if __name__ == "__main__":
    main()
