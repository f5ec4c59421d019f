"""SURVEY 8(f) N2 + N3: the trainer shell (npi_gnn_b200/train_shell.py) against the reference script
src/train_with_twoDataset.PY -- flags and defaults (:26-43), LR rule (:155-160), evaluation /
checkpoint cadence (:163,193-194,213-214), log line format (:168,172,199,203,219-221) -- and, on the
GPU, a whole run whose artefacts are cross-checked with the oracle."""
import os
import re

import numpy as np
import pytest
import torch

from tests.common import load_kat, npinter2_oracle_graph

REF_FLAGS = {        # src/train_with_twoDataset.PY:26-43  (flag -> default)
    "trainingName": None, "trainingDatasetName": None, "testingDatasetName": None, "inMemory": 1,
    "interactionDatasetName": "NPInter2", "fold": None, "epochNumber": 50, "hopNumber": 1,
    "node2vecWindowSize": 5, "initialLearningRate": 0.001, "l2WeightDecay": 0.001, "batchSize": 200,
}


def test_flags_and_defaults_match_reference_script():
    from npi_gnn_b200 import train_shell as ts
    a = ts.parse_args([])
    for k, v in REF_FLAGS.items():
        assert getattr(a, k) == v, k
    a = ts.parse_args("--trainingName t --trainingDatasetName A --testingDatasetName B --fold 3 --epochNumber 7 "
                      "--initialLearningRate 0.01 --l2WeightDecay 0.1 --batchSize 64 --hopNumber 2".split())
    assert (a.trainingName, a.fold, a.epochNumber, a.initialLearningRate, a.l2WeightDecay, a.batchSize, a.hopNumber) == \
        ("t", 3, 7, 0.01, 0.1, 64, 2)


@pytest.mark.reference
def test_flags_against_live_reference_source():
    from oracle import ref_import
    src = open(os.path.join(ref_import.REF_ROOT, "src", "train_with_twoDataset.PY"), encoding="utf-8").read()
    found = {}
    for line in src.splitlines():
        m = re.match(r"\s*parser\.add_argument\('--(\w+)'(.*)\)", line)
        if m:
            d = re.search(r"default=([^,)]+)", m.group(2))
            found[m.group(1)] = None if d is None else eval(d.group(1))
    assert found == REF_FLAGS


def test_lr_rule_cadence_and_log_format():
    from npi_gnn_b200 import train_shell as ts
    s = ts.LrOnLossIncrease(1e-3)
    lrs = [s.update(l) for l in (0.9, 0.8, 0.85, 0.85, 0.9, 0.7)]
    assert np.allclose(lrs, [1e-3, 1e-3, 0.95e-3, 0.95e-3, 0.95 ** 2 * 1e-3, 0.95 ** 2 * 1e-3])
    # every 5th epoch except the last one; the final evaluation happens after the loop
    assert [e for e in range(1, 51) if ts.should_evaluate(e, 50)] == [5, 10, 15, 20, 25, 30, 35, 40, 45]
    assert [e for e in range(1, 8) if ts.should_evaluate(e, 7)] == [5]
    # a line of the shipped log of project 1223_1, fold 0 (result/1223_1/log_0.txt) re-rendered from its numbers
    line = ts.metric_line("Epoch: {:03d}, testing dataset".format(15), (0.97, 0.9712, 0.968795, 0.97120, 0.94000421))
    assert line == ("Epoch: 015, testing dataset, Accuracy: 0.97000, Precision: 0.97120, Sensitivity: 0.96879, "
                    "Specificity: 0.97120, MCC: 0.94000")
    pat = re.compile(r"^(Epoch: \d{3}|result), (training|testing) dataset, Accuracy: \d\.\d{5}, Precision: \d\.\d{5}, "
                     r"Sensitivity: \d\.\d{5}, Specificity: \d\.\d{5}, MCC: -?\d\.\d{5}$")
    assert pat.match(line) and pat.match(ts.metric_line("result, training dataset", (1, 1, 1, 1, -0.5)))
    b = ts.BestByMcc()
    b.offer(5, (0.9, 0.8, 0.7, 0.6, 0.5)); b.offer(10, (0.1, 0.1, 0.1, 0.1, 0.4)); b.offer(15, (0.95, 0.9, 0.9, 0.9, 0.9))
    assert (b.epoch, b.mcc, b.acc) == (15, 0.9, 0.95)
    assert b.line() == "epoch: 15, MCC: 0.9, ACC: 0.95, Pre: 0.9, Sen: 0.9, Spe: 0.9"


def test_shipped_log_lines_match_the_format():
    """Every metric line of the reference's own logs that tests/golden/kat.json carries (the testing-dataset lines of
    result/1223_1/log_0.txt and result/1223_1_noKmer/log_0.txt, verbatim) is reproduced byte for byte by metric_line()."""
    from npi_gnn_b200 import train_shell as ts
    lines = [e["line"] for proj in load_kat()["confusion"].values() for e in proj.values()]
    n = 0
    for line in lines:
        m = re.match(r"^(Epoch: \d{3}, \w+ dataset|result, \w+ dataset), Accuracy: ([\d.]+), Precision: ([\d.]+), "
                     r"Sensitivity: ([\d.]+), Specificity: ([\d.]+), MCC: (-?[\d.]+)$", line)
        if m:
            assert ts.metric_line(m.group(1), tuple(float(v) for v in m.groups()[1:])) == line
            n += 1
    assert n == len(lines) and n >= 20


def test_run_refuses_cpu_and_bad_inmemory():
    from npi_gnn_b200 import NPIError, train_shell as ts
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(NPIError):
        ts.run(ts.parse_args(["--trainingName", "x", "--fold", "0"]))


def _datasets(tmp_path, h=1, n_train=600, n_test=200):
    from npi_gnn_b200 import LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory as DS
    d, g, mask = npinter2_oracle_graph()
    cannot = set(map(tuple, np.concatenate([d["test_pos"], d["test_neg"]]).tolist()))
    arr = dict(edges=d["edges"], is_rna=d["is_rna"], table=d["table"])
    ht, hs = n_train // 2, n_test // 2
    tr_pairs = np.concatenate([d["train_pos"][:ht], d["train_neg"][:ht]]).astype(np.int32)
    te_pairs = np.concatenate([d["test_pos"][:hs], d["test_neg"][:hs]]).astype(np.int32)
    tr = DS(str(tmp_path / "train"), h=h, set_allInteractionKey_cannotUse=cannot,
            arrays=dict(arr, pairs=tr_pairs, y=np.array([1] * ht + [0] * ht, dtype=np.int32)))
    te = DS(str(tmp_path / "test"), h=h, set_allInteractionKey_cannotUse=cannot,
            arrays=dict(arr, pairs=te_pairs, y=np.array([1] * hs + [0] * hs, dtype=np.int32)))
    return d, g, mask, cannot, tr, te, te_pairs


@pytest.mark.gpu
def test_whole_run_artefacts_and_oracle_cross_check(tmp_path):
    """7 epochs: log + checkpoints at 5 and 7 exist in the reference's layout; the logged testing
    metrics of epoch 5 and of the final model are reproduced by the CPU oracle from the saved
    state_dicts; the loss goes down; a second run into the same fold directory is refused."""
    from npi_gnn_b200 import train_shell as ts
    from oracle import khop_cwrap, net as onet
    d, g, mask, cannot, tr, te, te_pairs = _datasets(tmp_path)
    args = ts.parse_args(["--trainingName", "t1", "--trainingDatasetName", "train", "--testingDatasetName", "test", "--fold", "0",
                          "--epochNumber", "7", "--batchSize", "100", "--seed", "11", "--resultRoot", str(tmp_path / "result")])
    out = ts.run(args, echo=False, train_dataset=tr, test_dataset=te)
    assert out["backend"] == "fused" and len(out["losses"]) == 7 and out["losses"][-1] < out["losses"][0]
    assert sorted(os.listdir(out["model_dir"]), key=int) == ["5", "7"]
    text = open(out["log"], encoding="utf-8").read()
    lines = text.splitlines()
    assert lines[0].startswith("training dataset : traintesting dataset : testdatabase：NPInter2")
    assert "number of eopch ：7" in text and "L2 weight decay = 0.001" in text
    ev = [l for l in lines if l.startswith(("Epoch:", "result,"))]
    assert [l.split(", Accuracy")[0] for l in ev] == ["Epoch: 005, training dataset", "Epoch: 005, testing dataset",
                                                      "result, training dataset", "result, testing dataset"]
    assert any(l.startswith("epoch: ") for l in lines) and lines[-1].startswith("Time consuming:")
    # oracle on the saved checkpoints (reference state_dict names -> loads into the oracle's Net_1)
    for ck, line in (("5", ev[1]), ("7", ev[3])):
        sd = torch.load(os.path.join(out["model_dir"], ck))
        m = onet.Net_1(178)
        m.load_state_dict(sd)
        m.eval()
        y = np.array([1] * (len(te_pairs) // 2) + [0] * (len(te_pairs) // 2))
        c = khop_cwrap.collate_batch(g, mask, te_pairs, y, 1, d["table"])
        with torch.no_grad():
            pred = m(onet.batch_namespace(c)).argmax(1).numpy()
        TP = int(((pred == 1) & (y == 1)).sum()); FN = int(((pred == 0) & (y == 1)).sum())
        TN = int(((pred == 0) & (y == 0)).sum()); FP = int(((pred == 1) & (y == 0)).sum())
        from npi_gnn_b200 import metrics
        exp = ts.metric_line(line.split(", Accuracy")[0], metrics(TP, FN, TN, FP))
        got = [float(v) for v in re.findall(r": (-?\d\.\d{5})", line)]
        want = [float(v) for v in re.findall(r": (-?\d\.\d{5})", exp)]
        # a sample whose two logits tie within fp32 rounding may flip between the two stacks
        assert abs(got[0] - want[0]) <= 1.5 / len(te_pairs), (line, exp)
    with pytest.raises(Exception, match="Same fold"):
        ts.run(args, echo=False, train_dataset=tr, test_dataset=te)


@pytest.mark.gpu
def test_run_on_precomputed_pyg_cache_uses_module_route(tmp_path):
    """Datasets that only exist as the reference's processed/data.pt train through Net_1 + torch Adam."""
    from npi_gnn_b200 import LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory as DS, train_shell as ts
    d, g, mask, cannot, tr, te, te_pairs = _datasets(tmp_path, n_train=200, n_test=100)
    tr.write_pyg_cache(str(tmp_path / "data" / "A"))
    te.write_pyg_cache(str(tmp_path / "data" / "B"))
    args = ts.parse_args(["--trainingName", "t2", "--trainingDatasetName", "A", "--testingDatasetName", "B", "--fold", "1",
                          "--epochNumber", "6", "--batchSize", "50", "--seed", "5", "--dataRoot", str(tmp_path / "data"),
                          "--resultRoot", str(tmp_path / "result")])
    out = ts.run(args, echo=False)
    assert out["backend"] == "module" and out["losses"][-1] < out["losses"][0]
    assert sorted(os.listdir(out["model_dir"]), key=int) == ["5", "6"]
    sd = torch.load(os.path.join(out["model_dir"], "6"))
    assert list(sd.keys())[0] == "conv1.weight" and tuple(sd["conv1.weight"].shape) == (178, 128)
    assert 0.0 <= out["final_test"][0] <= 1.0
