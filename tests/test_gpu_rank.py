"""Ranking metrics on the GPU (npi_rank_curve, trainer.rank_metrics, Scorer.rank_metrics, --rankMetrics) against a
numpy oracle written here and, where it is installed, sklearn -- the library the reference's
src/compare_withKmer_noKmer.py computes ROC AUC and PR AUC with."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.common import fold0, load_ckpt, oracle_batches

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [7, 4095, 4097, 100003, 2081564]          # across the sort's 4,096-item tile, up to the config-5 sweep
REL = 1e-12


def oracle(s, y):
    """The curve and areas by np.unique + cumsum, twice_u by integer rank sums (midranks doubled)."""
    s = np.asarray(s, dtype=np.float32) + np.float32(0.0)          # -0.0 -> +0.0
    y = np.asarray(y, dtype=np.int64)
    order = np.argsort(-s, kind="stable")
    ss, yy = s[order], y[order]
    ends = np.nonzero(np.r_[ss[1:] != ss[:-1], True])[0]
    tps = np.cumsum(yy == 1)[ends]
    fps = ends + 1 - tps
    n_pos, n_neg = int(tps[-1]), int(fps[-1])
    _, inv, cnt = np.unique(s, return_inverse=True, return_counts=True)
    lo = np.cumsum(cnt) - cnt
    two_mid = (2 * lo + cnt + 1).astype(np.int64)                    # twice the 1-based midrank of each distinct score
    twice_u = int(two_mid[inv][y == 1].sum()) - n_pos * (n_pos + 1)
    prec = tps / (tps + fps)
    dt = np.diff(np.r_[0, tps])
    prev = np.r_[1.0, prec[:-1]]
    return dict(thresholds=ss[ends], tps=tps, fps=fps, n_pos=n_pos, n_neg=n_neg, twice_u=twice_u,
                auroc=twice_u / (2.0 * n_pos * n_neg), ap=float((dt * prec).sum() / n_pos),
                pr_auc_trapz=float(0.5 * (dt * (prec + prev)).sum() / n_pos))


def _case(n, seed):
    rng = np.random.default_rng(seed)
    s = (rng.integers(-40, 41, n) / 8.0).astype(np.float32)          # coarse grid: heavy ties
    s[rng.random(n) < 0.05] = -0.0
    y = (rng.random(n) < 0.3).astype(np.int32)
    y[0], y[1] = 1, 0
    return s, y


def _gpu(s, y, curve=True):
    from npi_gnn_b200.trainer import rank_metrics
    r = rank_metrics(torch.as_tensor(s).cuda(), torch.as_tensor(y).cuda(), curve=curve)
    return {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in r.items()}


def _check_vs_oracle(r, o):
    T = len(o["tps"])
    assert (r["n_pos"], r["n_neg"], r["twice_u"], len(r["thresholds"])) == (o["n_pos"], o["n_neg"], o["twice_u"], T)
    assert np.array_equal(r["thresholds"], o["thresholds"])
    assert np.array_equal(r["tpr"], o["tps"] / o["n_pos"]) and np.array_equal(r["fpr"], o["fps"] / o["n_neg"])
    assert np.array_equal(r["precision"], o["tps"] / (o["tps"] + o["fps"])) and np.array_equal(r["recall"], r["tpr"])
    assert r["auroc"] == o["auroc"]
    for k in ("ap", "pr_auc_trapz"):
        assert abs(r[k] - o[k]) <= REL * abs(o[k]), (k, r[k], o[k])


# ----------------------------------------------------------------------------- hand cases
def test_all_scores_tied():
    y = np.array([1, 0, 1, 0, 0, 0, 1, 0, 0, 0], dtype=np.int32)
    r = _gpu(np.full(10, 0.25, dtype=np.float32), y)
    assert r["auroc"] == 0.5 and abs(r["ap"] - 0.3) < 1e-15 and len(r["thresholds"]) == 1
    assert r["twice_u"] == 3 * 7


def test_perfect_and_reversed_separation():
    s = np.arange(20, dtype=np.float32)
    y = (s >= 12).astype(np.int32)
    r = _gpu(s, y)
    assert r["auroc"] == 1.0 and r["ap"] == 1.0 and r["pr_auc_trapz"] == 1.0
    r = _gpu(-s, y)
    assert r["auroc"] == 0.0 and r["twice_u"] == 0


def test_signed_zeros_are_one_threshold():
    s = np.array([-0.0, 0.0, 1.0, -0.0, 0.0], dtype=np.float32)
    y = np.array([1, 0, 1, 0, 1], dtype=np.int32)
    r = _gpu(s, y)
    assert list(r["thresholds"]) == [1.0, 0.0] and list(r["tpr"]) == [1 / 3, 1.0] and list(r["fpr"]) == [0.0, 1.0]
    _check_vs_oracle(r, oracle(s, y))


def test_infinite_scores():
    s = np.array([np.inf, 1.0, -np.inf, np.inf, 0.0, -np.inf], dtype=np.float32)
    y = np.array([1, 0, 0, 1, 1, 0], dtype=np.int32)
    r = _gpu(s, y)
    assert list(r["thresholds"]) == [np.inf, 1.0, 0.0, -np.inf]
    _check_vs_oracle(r, oracle(s, y))


def test_two_items_and_one_class():
    from npi_gnn_b200.trainer import rank_metrics
    r = _gpu(np.array([0.3, 0.7], dtype=np.float32), np.array([0, 1], dtype=np.int32))
    assert (r["auroc"], r["ap"], r["n_pos"], r["n_neg"]) == (1.0, 1.0, 1, 1)
    with pytest.raises(ValueError):
        rank_metrics(torch.tensor([0.5], device="cuda"), torch.tensor([1], dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError):
        rank_metrics(torch.rand(50, device="cuda"), torch.zeros(50, dtype=torch.int32, device="cuda"))


def test_nan_scores_and_bad_labels_raise():
    from npi_gnn_b200 import NPIError
    from npi_gnn_b200.trainer import rank_metrics
    s = torch.rand(9000, device="cuda")
    y = (torch.arange(9000, device="cuda") % 3 == 0).to(torch.int32)
    s2 = s.clone(); s2[8500] = float("nan")
    with pytest.raises(NPIError, match="NaN"):
        rank_metrics(s2, y)
    y2 = y.clone(); y2[4100] = 2
    with pytest.raises(NPIError, match="label"):
        rank_metrics(s, y2)
    y2[4100] = -1
    with pytest.raises(NPIError, match="label"):
        rank_metrics(s, y2)
    assert rank_metrics(s, y)["n_pos"] == 3000


def test_argument_checks():
    from npi_gnn_b200 import NPIError, ops
    s = torch.rand(5000, device="cuda")
    y = torch.zeros(5000, dtype=torch.int32, device="cuda")
    res = torch.zeros(7, dtype=torch.int64, device="cuda")
    small = torch.empty(ops.rank_workspace_bytes(5000) - 1, dtype=torch.uint8, device="cuda")
    with pytest.raises(NPIError, match="workspace"):
        ops.rank_curve(s, y, res[:4], res[4:6].view(torch.float64), res[6:7].view(torch.int32)[:1], small)
    ws = torch.empty(ops.rank_workspace_bytes(5000), dtype=torch.uint8, device="cuda")
    with pytest.raises(NPIError, match="rank_curve"):
        ops.rank_curve(s[:0], y[:0], res[:4], res[4:6].view(torch.float64), res[6:7].view(torch.int32)[:1], ws)
    with pytest.raises(NPIError, match="float32"):
        ops.rank_curve(s.double(), y, res[:4], res[4:6].view(torch.float64), res[6:7].view(torch.int32)[:1], ws)


# ----------------------------------------------------------------------------- random cases
@pytest.mark.parametrize("n", SIZES)
def test_random_ties_vs_numpy_oracle(n):
    s, y = _case(n, seed=n)
    _check_vs_oracle(_gpu(s, y), oracle(s, y))


@pytest.mark.parametrize("n", SIZES)
def test_random_ties_vs_sklearn(n):
    skm = pytest.importorskip("sklearn.metrics")
    s, y = _case(n, seed=n)
    r = _gpu(s, y)
    fpr, tpr, thr = skm.roc_curve(y, s, drop_intermediate=False)
    assert np.array_equal(r["thresholds"], thr[1:]) and np.array_equal(r["fpr"], fpr[1:]) and np.array_equal(r["tpr"], tpr[1:])
    p, rc, _ = skm.precision_recall_curve(y, s)
    assert np.array_equal(r["precision"], p[:-1][::-1]) and np.array_equal(r["recall"], rc[:-1][::-1])
    for got, want in ((r["auroc"], skm.roc_auc_score(y, s)), (r["ap"], skm.average_precision_score(y, s)),
                      (r["pr_auc_trapz"], skm.auc(rc, p))):
        assert abs(got - want) <= REL * abs(want), (got, want)


# ----------------------------------------------------------------------------- determinism, capture
def _raw(s, y):
    from npi_gnn_b200 import ops
    n = s.numel()
    res = torch.zeros(7, dtype=torch.int64, device="cuda")
    thr = torch.empty(n, dtype=torch.float32, device="cuda")
    tps = torch.empty(n, dtype=torch.int32, device="cuda")
    fps = torch.empty(n, dtype=torch.int32, device="cuda")
    ws = torch.empty(ops.rank_workspace_bytes(n), dtype=torch.uint8, device="cuda")
    return res, thr, tps, fps, ws


def _run_raw(s, y, bufs):
    from npi_gnn_b200 import ops
    res, thr, tps, fps, ws = bufs
    ops.rank_curve(s, y, res[:4], res[4:6].view(torch.float64), res[6:7].view(torch.int32)[:1], ws, thr, tps, fps)


def _curve_of(bufs):
    """summary + areas (as int64 bits), status, and the curve: everything the call writes."""
    res, thr, tps, fps, _ = bufs
    T = int(res[2])
    return res[:6].clone(), res[6:7].view(torch.int32)[:1].clone(), thr[:T].clone(), tps[:T].clone(), fps[:T].clone()


def _same(a, b):
    return all(torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int32) if y.dtype == torch.float32 else y) for x, y in zip(a, b))


def test_bit_identical_on_rerun_and_under_permutation():
    s_np, y_np = _case(300007, seed=5)
    s, y = torch.as_tensor(s_np).cuda(), torch.as_tensor(y_np).cuda()
    bufs = _raw(s, y)
    _run_raw(s, y, bufs)
    first = _curve_of(bufs)
    bufs[0].fill_(-1)
    _run_raw(s, y, bufs)
    assert _same(first, _curve_of(bufs))
    perm = torch.as_tensor(np.random.default_rng(9).permutation(len(s_np))).cuda()
    _run_raw(s[perm].contiguous(), y[perm].contiguous(), bufs)
    assert _same(first, _curve_of(bufs))
    assert int(first[1][0]) == 0 and int(first[0][0]) == int(y_np.sum())


def test_cuda_graph_capture_and_replay_on_new_inputs():
    n = 50000
    s0, y0 = _case(n, seed=1)
    s1, y1 = _case(n, seed=2)
    s, y = torch.as_tensor(s0).cuda(), torch.as_tensor(y0).cuda()
    bufs = _raw(s, y)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _run_raw(s, y, bufs)                          # warm-up outside capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _run_raw(s, y, bufs)
    s.copy_(torch.as_tensor(s1)); y.copy_(torch.as_tensor(y1))
    bufs[0].fill_(-1)
    g.replay()
    torch.cuda.synchronize()
    eager = _raw(s, y)
    _run_raw(torch.as_tensor(s1).cuda(), torch.as_tensor(y1).cuda(), eager)
    assert _same(_curve_of(bufs), _curve_of(eager))
    o = oracle(s1, y1)
    assert int(bufs[0][3]) == o["twice_u"]


# ----------------------------------------------------------------------------- Scorer on the real fold-0 test set
def test_scorer_rank_metrics_on_npinter2_fold0():
    from npi_gnn_b200.trainer import Scorer
    from oracle import net as onet
    d, og, omask, pairs, ys, ps, params = fold0()
    sc = Scorer(ps, params, batch_size=200)
    r = sc.rank_metrics(curve=True)
    p = sc.probabilities().cpu().numpy()
    o = oracle(p, ys)
    _check_vs_oracle({k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in r.items()}, o)
    skm = None
    try:
        import sklearn.metrics as skm
    except ImportError:
        pass
    if skm is not None:
        assert abs(r["auroc"] - skm.roc_auc_score(ys, p)) <= REL and abs(r["ap"] - skm.average_precision_score(ys, p)) <= REL
    assert r["confusion"] == sc.confusion()
    # the CPU oracle's probabilities: fp32 rounding may flip near-ties, each flip moves AUROC by <= 1 / (n_pos n_neg)
    m = onet.Net_1(ps.graph.F)
    m.load_state_dict(load_ckpt("ckpt_1223_1_15.npz"))
    m.eval()
    with torch.no_grad():
        po = np.concatenate([torch.exp(m(onet.batch_namespace(c))[:, 1]).numpy()
                             for c in oracle_batches(pairs, ys.astype(np.int64), 1, d["table"], og, omask)])
    assert abs(r["auroc"] - oracle(po, ys)["auroc"]) <= 1e-5
    # a shuffled index view: labels follow the view, every metric bit for bit the same
    perm = np.random.default_rng(3).permutation(len(pairs))
    r2 = Scorer(ps, params, batch_size=200, index=perm).rank_metrics(curve=True)
    for k in ("auroc", "ap", "pr_auc_trapz", "n_pos", "n_neg", "twice_u", "confusion"):
        assert r2[k] == r[k], k
    for k in ("thresholds", "fpr", "tpr", "precision", "recall"):
        assert torch.equal(r2[k], r[k]), k


def test_scorer_rank_metrics_needs_a_process_group_when_sharded():
    from npi_gnn_b200 import NPIError
    from npi_gnn_b200.trainer import Scorer
    d, og, omask, pairs, ys, ps, params = fold0()
    with pytest.raises(NPIError, match="process group"):
        Scorer(ps, params, batch_size=200, world_size=2, rank=0).rank_metrics()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_rank_metrics_two_gpus_match_one():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29637", os.path.join(ROOT, "tests", "scorer_dp_worker.py"),
           "rank_metrics"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stderr[-3000:]
    assert "RANK_DP_OK" in out.stdout


# ----------------------------------------------------------------------------- trainer shell
RANK_LINE = re.compile(r"^(Epoch: \d{3}|result), testing dataset, AUROC: \d\.\d{5}, AP: \d\.\d{5}, PR-AUC\(trapz\): \d\.\d{5}$")


def _shell_pair(tmp_path, argv, **kw):
    """The same seeded run without and with --rankMetrics 1: (log lines, checkpoint dir) of each."""
    from npi_gnn_b200 import train_shell as ts
    runs = []
    for flag, name in ((0, "plain"), (1, "ranked")):
        args = ts.parse_args(argv + ["--trainingName", name, "--resultRoot", str(tmp_path / "result"), "--rankMetrics", str(flag)])
        out = ts.run(args, echo=False, **kw)
        runs.append((open(out["log"], encoding="utf-8").read().splitlines(), out["model_dir"]))
    return runs


def _check_shell_pair(runs):
    (plain, dir0), (ranked, dir1) = runs
    ranked_lines = [l for l in ranked if ", AUROC: " in l]
    assert ranked_lines and all(RANK_LINE.match(l) for l in ranked_lines)
    for i, l in enumerate(ranked):
        if l.startswith(("Epoch:", "result,")) and "testing dataset, Accuracy" in l:
            assert RANK_LINE.match(ranked[i + 1]) and ranked[i + 1].split(", AUROC")[0] == l.split(", Accuracy")[0]
            assert ", AUROC: " not in ranked[i + 2]
    strip = lambda ls: [l for l in ls if ", AUROC: " not in l and not l.startswith("Time consuming")]
    assert strip(ranked) == strip(plain)
    assert not any(", AUROC: " in l for l in plain)
    assert sorted(os.listdir(dir0)) == sorted(os.listdir(dir1))
    for f in os.listdir(dir0):
        assert open(os.path.join(dir0, f), "rb").read() == open(os.path.join(dir1, f), "rb").read(), f


def test_train_shell_rank_metrics_fused_route(tmp_path):
    from tests.test_train_shell import _datasets
    d, g, mask, cannot, tr, te, te_pairs = _datasets(tmp_path)
    runs = _shell_pair(tmp_path, ["--trainingDatasetName", "train", "--testingDatasetName", "test", "--fold", "0",
                                  "--epochNumber", "7", "--batchSize", "100", "--seed", "11"], train_dataset=tr, test_dataset=te)
    _check_shell_pair(runs)
    assert sum(", AUROC: " in l for l in runs[1][0]) == 2


def test_train_shell_rank_metrics_module_route(tmp_path):
    from tests.test_train_shell import _datasets
    d, g, mask, cannot, tr, te, te_pairs = _datasets(tmp_path, n_train=200, n_test=100)
    tr.write_pyg_cache(str(tmp_path / "data" / "A"))
    te.write_pyg_cache(str(tmp_path / "data" / "B"))
    runs = _shell_pair(tmp_path, ["--trainingDatasetName", "A", "--testingDatasetName", "B", "--fold", "1", "--epochNumber", "6",
                                  "--batchSize", "50", "--seed", "5", "--dataRoot", str(tmp_path / "data")])
    _check_shell_pair(runs)
    assert sum(", AUROC: " in l for l in runs[1][0]) == 2
