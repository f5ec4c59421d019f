"""Time the filtered per-node ranking on the GPU and write one JSON record (device name and power limit read in the same
run).

    python tools/partner_rank_time.py [--out FILE] [--reps 100]

  - trainer.group_rank_metrics over the 2,081,564 pairs of the config-5 sweep (every RNA x protein pair of the
    NPInter2-shaped graph, RNA-major), grouped by RNA (4,636 groups of 449 pairs) and by protein (449 groups of 4,636),
    node serials as group ids (num_groups = 5,085 nodes).  Queries: the pairs of synth.npinter2_shaped()["pos"] (label
    1, 9,905 of them); every other pair is a competitor.  Scores: seeded uniform probabilities rounded to a 1e-4 grid,
    so that ties occur.  CUDA events over --reps calls after warm-up: the whole call (output and workspace allocation,
    the launches, the per-group AUC, its one synchronising read) one at a time, and npi_group_rank alone back to back
    into preallocated buffers.  Working set ~60 MB (inputs, sort buffers, scan), not flushed from the 126 MB L2 between
    calls.
  - the host route it replaces: device-to-host copy of the scores, then per group a numpy ranking of every query among
    the group's competitors (lexsort of (group, score) keys + searchsorted) and the summary; its above / tied counts
    are checked equal to the GPU's.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from npi_gnn_b200 import ops, synth  # noqa: E402
from npi_gnn_b200.trainer import group_rank_metrics  # noqa: E402
from rank_time import device_info  # noqa: E402  (tools/rank_time.py, next to this script)
from topk_time import events_ms  # noqa: E402

HITS = (1, 3, 10)


def host_rank(s_dev, y, grp, G):
    """The numpy route: copy, (group, score) keys, competitors lexsorted, queries located by searchsorted."""
    s = s_dev.cpu().numpy() + np.float32(0.0)                         # -0.0 -> +0.0
    q, c = y == 1, y == 0
    cg, cs = grp[c].astype(np.int64), s[c]
    order = np.lexsort((cs, cg))                                    # group, then ascending score
    cg, cs = cg[order], cs[order]
    bounds = np.searchsorted(cg, np.arange(G + 1))
    qg, qs = grp[q].astype(np.int64), s[q]
    # per query: competitors of its group at or below its score, found group by group on the sorted slice
    above = np.empty(len(qg), dtype=np.int64)
    tied = np.empty(len(qg), dtype=np.int64)
    qorder = np.argsort(qg, kind="stable")
    qb = np.searchsorted(qg[qorder], np.arange(G + 1))
    for g in np.nonzero(qb[1:] > qb[:-1])[0]:
        sl = cs[bounds[g]:bounds[g + 1]]
        idx = qorder[qb[g]:qb[g + 1]]
        lo, hi = np.searchsorted(sl, qs[idx], "left"), np.searchsorted(sl, qs[idx], "right")
        above[idx], tied[idx] = len(sl) - hi, hi - lo
    n_neg = bounds[1:] - bounds[:-1]
    ranked = n_neg[qg] > 0
    twice_rank = 2 * above[ranked] + tied[ranked] + 2
    nq = int(ranked.sum())
    return above, tied, dict(mrr=float(np.sum(2.0 / twice_rank)) / nq,
                             hits={k: int((twice_rank <= 2 * k).sum()) / nq for k in HITS}, n_queries=nq)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=100)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "partner_rank_time.py measures on the GPU"
    torch.cuda.set_device(0)
    rec = {"tool": "tools/partner_rank_time.py", **device_info()}
    d = synth.npinter2_shaped()
    allp = synth.all_candidate_pairs(d)
    V = len(d["is_rna"])
    pos = np.asarray(d["pos"])
    y_np = np.isin(allp[:, 0].astype(np.int64) * V + allp[:, 1], pos[:, 0].astype(np.int64) * V + pos[:, 1]).astype(np.int32)
    rng = np.random.default_rng(20240602)
    s = torch.as_tensor(np.round(rng.random(len(allp)), 4).astype(np.float32)).cuda()
    y = torch.as_tensor(y_np).cuda()
    n = len(allp)
    rec.update(n=n, num_groups=V, queries=int(y_np.sum()), hits=list(HITS))
    cases = {}
    for name, col in (("per_rna", 0), ("per_protein", 1)):
        grp_np = np.ascontiguousarray(allp[:, col])
        grp = torch.as_tensor(grp_np).cuda()
        i32 = dict(dtype=torch.int32, device="cuda")
        bufs = (torch.empty(V, **i32), torch.empty(V, **i32), torch.empty(V, dtype=torch.int64, device="cuda"),
                torch.empty(3 + len(HITS), dtype=torch.int64, device="cuda"), torch.empty(1, dtype=torch.float64, device="cuda"),
                torch.empty(1, **i32), torch.empty(ops.group_rank_workspace_bytes(n, V), dtype=torch.uint8, device="cuda"))
        for _ in range(5):
            group_rank_metrics(s, y, grp, V, HITS)
            ops.group_rank(s, y, grp, V, HITS, *bufs)
        torch.cuda.synchronize()
        call_med, call_min, _ = events_ms(lambda: group_rank_metrics(s, y, grp, V, HITS), args.reps)
        raw_med, raw_min, raw_b2b = events_ms(lambda: ops.group_rank(s, y, grp, V, HITS, *bufs), args.reps)
        r = group_rank_metrics(s, y, grp, V, HITS, per_item=True)
        host_ms = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            above, tied, hs = host_rank(s, y_np, grp_np, V)
            host_ms.append((time.perf_counter() - t0) * 1e3)
        q = y_np == 1
        equal = bool(np.array_equal(r["above"].cpu().numpy()[q], above) and np.array_equal(r["tied"].cpu().numpy()[q], tied)
                     and r["n_queries"] == hs["n_queries"] and r["hits"] == hs["hits"])
        cases[name] = {
            "groups": int((np.bincount(grp_np, minlength=V) > 0).sum()), "reps": args.reps,
            "mrr": r["mrr"], "hits": {str(k): v for k, v in r["hits"].items()}, "auc_macro": r["auc_macro"],
            "n_queries": r["n_queries"], "n_unranked": r["n_unranked"], "n_groups_scored": r["n_groups_scored"],
            "group_rank_metrics_ms_median": call_med, "group_rank_metrics_ms_min": call_min,
            "group_rank_ms_median_isolated": raw_med, "group_rank_ms_min_isolated": raw_min,
            "group_rank_ms_back_to_back": raw_b2b,
            "numpy_host_ms_median": float(np.median(host_ms)), "numpy_host_ms_min": float(np.min(host_ms)),
            "mrr_rel_diff_to_numpy": abs(r["mrr"] - hs["mrr"]) / hs["mrr"],
            "equal_to_numpy": equal}
    rec["group_rank_metrics"] = cases
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
