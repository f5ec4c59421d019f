"""Known-answer tests that PIN the oracle (SURVEY.md 0.5): shipped checkpoints + the metric
lines of result/1223_1*/log_0.txt + the case-study partitions, all carried as fixtures in
tests/golden (tools/make_golden.py)."""
import math

import numpy as np
import pytest
import torch

from oracle import net as onet
from tests.common import load_ckpt, load_kat, npinter2_oracle_graph, oracle_batches


def _test_batches(no_kmer=False):
    d, g, mask = npinter2_oracle_graph()
    table = d["table"][:, :64].copy() if no_kmer else d["table"]
    pairs = np.concatenate([d["test_pos"], d["test_neg"]])
    ys = np.concatenate([np.ones(len(d["test_pos"]), dtype=np.int64), np.zeros(len(d["test_neg"]), dtype=np.int64)])
    perm = np.random.default_rng(0).permutation(len(pairs))
    return [onet.batch_namespace(c) for c in oracle_batches(pairs[perm], ys[perm], 1, table, g, mask)]


@pytest.mark.parametrize("proj,ep", [("1223_1", 5), ("1223_1", 15), ("1223_1", 30), ("1223_1", 50),
                                     ("1223_1_noKmer", 20), ("1223_1_noKmer", 35), ("1223_1_noKmer", 50)])
def test_confusion_matrix_kat(proj, ep):
    torch.set_flush_denormal(True)
    no_kmer = proj.endswith("noKmer")
    m = onet.Net_1(65 if no_kmer else 178)
    m.load_state_dict(load_ckpt("ckpt_%s_%d.npz" % (proj, ep)))
    exp = load_kat()["confusion"][proj][str(ep)]
    TP, FN, TN, FP = onet.confusion(m, _test_batches(no_kmer))
    assert (TP, FN, TN, FP) == (exp["TP"], exp["FN"], exp["TN"], exp["FP"])


@pytest.mark.parametrize("thr", ["0.5", "0.95"])
def test_case_study_kat(thr):
    """src/case_study_negativeSample.py:235-253,339-355: batch-size-1 eval forward per test
    negative, positive iff exp(logp[1]) > threshold."""
    torch.set_flush_denormal(True)
    d, g, mask = npinter2_oracle_graph()
    exp = load_kat()["case_study"][thr]
    m = onet.Net_1(178)
    m.load_state_dict(load_ckpt(exp["ckpt"]))
    m.eval()
    pairs = d["test_neg"]
    got = []
    with torch.no_grad():
        for c in oracle_batches(pairs, np.zeros(len(pairs), dtype=np.int64), 1, d["table"], g, mask, 256):
            p1 = torch.exp(m(onet.batch_namespace(c))[:, 1])
            off = len(got)
            got.extend(p1.tolist())
    pos = sorted([list(map(int, pairs[i])) for i, p in enumerate(got) if p > float(thr)])
    assert pos == exp["positives"]


@pytest.mark.reference
@pytest.mark.parametrize("proj", ["1223_1", "1223_1_noKmer"])
def test_live_every_shipped_fold0_checkpoint(proj):
    """The shipped checkpoints of fold 0 (result/<proj>/model_0_fold/{5..50}) against the
    `testing dataset` lines of result/<proj>/log_0.txt (tests/golden/kat.json carries the ten implied
    confusion matrices per variant): exact known answers computed by the authors' PyG-1.4.2 stack.
    The checkpoints are read from the reference tree, so this runs where that tree is (ref_import.REF_ROOT); seven
    travel as fixtures (test_confusion_matrix_kat), four more per variant are checked here by
    default and all ten with NPI_ALL_KATS=1 (all twenty reproduce exactly)."""
    import os
    from oracle import ref_import
    root = os.path.join(ref_import.REF_ROOT, "result", proj, "model_0_fold")
    if not os.path.isdir(root):
        pytest.skip("reference tree not present")
    torch.set_flush_denormal(True)
    no_kmer = proj.endswith("noKmer")
    batches = _test_batches(no_kmer)
    kat = load_kat()["confusion"][proj]
    assert len(kat) == 10
    # default: the epochs no fixture carries; NPI_ALL_KATS=1: all ten
    epochs = sorted(map(int, kat)) if os.environ.get("NPI_ALL_KATS") else (10, 20, 30, 40)
    for ep in epochs:
        sd = torch.load(os.path.join(root, str(ep)), map_location="cpu", weights_only=False)
        sd = sd if isinstance(sd, dict) else sd.state_dict()
        m = onet.Net_1(65 if no_kmer else 178)
        m.load_state_dict(sd)
        exp = kat[str(ep)]
        assert onet.confusion(m, batches) == (exp["TP"], exp["FN"], exp["TN"], exp["FP"]), (proj, ep)


@pytest.mark.reference
@pytest.mark.parametrize("fold", [1, 2, 3, 4])
def test_live_other_folds_of_project_1223_1(fold):
    """Folds 1-4 of project 1223_1 are shipped too (key sets, per-fold node2vec embedding, ten
    checkpoints and a log per fold and feature variant): the fold's graph and table are rebuilt from
    the raw files (oracle/refdata.py), the test subgraphs extracted and two checkpoints per variant
    compared with their log lines -- 16 more exact known answers (all ten epochs per fold, 80, with
    NPI_ALL_KATS=1).  Needs the reference tree (ref_import.REF_ROOT)."""
    import os
    from oracle import khop, khop_cwrap, ref_import, refdata
    ref = ref_import.REF_ROOT
    if not os.path.isdir(os.path.join(ref, "result", "1223_1", "model_%d_fold" % fold)):
        pytest.skip("reference tree not present")
    torch.set_flush_denormal(True)
    ds, keys, table = refdata.load_project(ref, "1223_1", "NPInter2", fold)
    g = khop.build_csr(ds.edges, ds.is_rna)
    cannot = keys["set_interactionKey_test"] + keys["set_negativeInteractionKey_test"]      # src/generate_dataset.py:297-299
    mask = khop.mask_from_keys(g, [tuple(k) for k in cannot])
    tp = np.asarray(keys["set_interactionKey_test"], dtype=np.int32)
    tn = np.asarray(keys["set_negativeInteractionKey_test"], dtype=np.int32)
    pairs = np.concatenate([tp, tn])
    ys = np.concatenate([np.ones(len(tp), dtype=np.int64), np.zeros(len(tn), dtype=np.int64)])
    epochs = range(5, 55, 5) if os.environ.get("NPI_ALL_KATS") else (30, 50)
    for proj in ("1223_1", "1223_1_noKmer"):
        no_kmer = proj.endswith("noKmer")
        tab = table[:, :64].copy() if no_kmer else table
        batches = [onet.batch_namespace(c) for c in oracle_batches(pairs, ys, 1, tab, g, mask)]
        kat = refdata.parse_metric_log(os.path.join(ref, "result", proj, "log_%d.txt" % fold), len(tp), len(tn))
        for ep in epochs:
            sd = torch.load(os.path.join(ref, "result", proj, "model_%d_fold" % fold, str(ep)), map_location="cpu", weights_only=False)
            m = onet.Net_1(65 if no_kmer else 178)
            m.load_state_dict(sd)
            exp = kat[ep]
            assert onet.confusion(m, batches) == (exp["TP"], exp["FN"], exp["TN"], exp["FP"]), (proj, fold, ep)
