"""Time the ranking metrics on the GPU and write one JSON record (device name and power limit read in the same run).

    python tools/rank_time.py [--out FILE] [--reps 50]

  - npi_rank_curve (17 launches, curve arrays requested) timed with CUDA events over --reps calls after warm-up, at
    n = 4,166 (the size of the NPInter2 fold-0 test set: 2,083 positive + 2,083 negative candidate pairs, seeded) and
    n = 2,081,564 (every RNA x protein pair of the NPInter2-shaped graph, config 5).  Labels: 1 for the pairs in
    synth.npinter2_shaped()["pos"], 0 for the other candidate pairs.  Scores: seeded logits (+2 for positives) rounded
    to a 1e-4 grid, so that ties are realistic.  Working set of the large case: ~110 MB (inputs, sort buffers, curve),
    not flushed from the 126 MB L2 between calls.
  - for the same arrays, sklearn's roc_auc_score + average_precision_score on the CPU including the device-to-host copy,
    if sklearn imports (else the record says it is absent).
  - one full 1-GPU Scorer sweep of the config-5 pairs (h = 2, 2,048 pairs per forward, fixed random weights):
    probabilities() alone against rank_metrics(), alternated, best of --sweeps each.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from npi_gnn_b200 import ops, synth  # noqa: E402
from npi_gnn_b200.engine import FlatParams  # noqa: E402
from npi_gnn_b200.graph import BipartiteGraph, PairSet  # noqa: E402
from npi_gnn_b200.trainer import Scorer, rank_metrics  # noqa: E402


def device_info():
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        out["nvidia_smi"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError) as ex:
        out["nvidia_smi"] = "unavailable: %s" % ex
    return out


def time_rank_curve(s, y, reps):
    n = s.numel()
    res = torch.zeros(7, dtype=torch.int64, device="cuda")
    thr = torch.empty(n, dtype=torch.float32, device="cuda")
    tps = torch.empty(n, dtype=torch.int32, device="cuda")
    fps = torch.empty(n, dtype=torch.int32, device="cuda")
    ws = torch.empty(ops.rank_workspace_bytes(n), dtype=torch.uint8, device="cuda")

    def call():
        ops.rank_curve(s, y, res[:4], res[4:6].view(torch.float64), res[6:7].view(torch.int32)[:1], ws, thr, tps, fps)
    for _ in range(5):
        call()
    torch.cuda.synchronize()
    per = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); call(); e1.record()
        e1.synchronize()
        per.append(e0.elapsed_time(e1))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        call()
    e1.record()
    torch.cuda.synchronize()
    return {"n": n, "reps": reps, "ms_per_call_back_to_back": e0.elapsed_time(e1) / reps,
            "ms_per_call_median_isolated": float(np.median(per)), "ms_per_call_min_isolated": float(np.min(per)),
            "n_thresholds": int(res[2]), "workspace_bytes": ws.numel()}


def time_sklearn(s, y, reps):
    try:
        import sklearn
        from sklearn.metrics import average_precision_score, roc_auc_score
    except ImportError as ex:
        return {"absent": "sklearn does not import: %s" % ex}
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sh, yh = s.cpu().numpy(), y.cpu().numpy()
        auc, ap = roc_auc_score(yh, sh), average_precision_score(yh, sh)
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"sklearn": sklearn.__version__, "reps": reps, "ms_median": float(np.median(ts)), "ms_min": float(np.min(ts)),
            "auroc": auc, "ap": ap}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--sweeps", type=int, default=2)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "rank_time.py measures on the GPU"
    torch.cuda.set_device(0)
    rec = {"tool": "tools/rank_time.py", **device_info()}
    d = synth.npinter2_shaped()
    allp = synth.all_candidate_pairs(d)
    n_prot = int((d["is_rna"] == 0).sum())
    r_of = np.cumsum(d["is_rna"].astype(np.int64)) - 1      # RNA serial -> row of the RNA-major candidate list
    p_of = np.cumsum((d["is_rna"] == 0).astype(np.int64)) - 1
    labels = np.zeros(len(allp), dtype=np.int32)
    labels[r_of[d["pos"][:, 0]] * n_prot + p_of[d["pos"][:, 1]]] = 1
    assert np.array_equal(allp[r_of[d["pos"][:, 0]] * n_prot + p_of[d["pos"][:, 1]]], d["pos"])
    rng = np.random.default_rng(20240601)
    logits = np.round(rng.standard_normal(len(allp)) + 2.0 * labels, 4).astype(np.float32)
    small = np.concatenate([rng.choice(np.nonzero(labels == 1)[0], 2083, replace=False),
                            rng.choice(np.nonzero(labels == 0)[0], 2083, replace=False)])
    cases = {}
    for name, idx in (("fold0_test_size", small), ("config5_sweep", np.arange(len(allp)))):
        s = torch.as_tensor(logits[idx]).cuda()
        y = torch.as_tensor(labels[idx]).cuda()
        c = time_rank_curve(s, y, args.reps)
        r = rank_metrics(s, y)
        c.update(auroc=r["auroc"], ap=r["ap"], pr_auc_trapz=r["pr_auc_trapz"], n_pos=r["n_pos"])
        c["sklearn_cpu"] = time_sklearn(s, y, 3 if len(idx) > 100000 else 20)
        cases[name] = c
    rec["rank_curve"] = cases
    # the metric's extra cost on a whole scoring sweep
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda:0")
    g.set_mask(synth.masked_pairs(d))
    ps = PairSet(g, allp, labels, h=2)
    params = FlatParams(g.F, "cuda:0").init_reference(torch.Generator().manual_seed(0))
    sc = Scorer(ps, params, batch_size=2048)
    out = torch.empty(len(allp), dtype=torch.float32, device="cuda")

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); res = fn(); e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), res
    timed(lambda: sc.probabilities(out))                   # graph capture + warm caches
    timed(lambda: sc.rank_metrics())
    prob_ms, rank_ms = [], []
    for _ in range(args.sweeps):
        prob_ms.append(timed(lambda: sc.probabilities(out))[0])
        ms, r = timed(lambda: sc.rank_metrics())
        rank_ms.append(ms)
    rec["scorer_sweep"] = {"pairs": len(allp), "h": 2, "batch": 2048, "sweeps": args.sweeps,
                           "probabilities_ms": prob_ms, "rank_metrics_ms": rank_ms,
                           "extra_ms_best": min(rank_ms) - min(prob_ms), "auroc": r["auroc"], "confusion": r["confusion"],
                           "note": "device events around the whole call, including rank_metrics' one synchronising read"}
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
