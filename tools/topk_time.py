"""Time the per-group top-k on the GPU and write one JSON record (device name and power limit read in the same run).

    python tools/topk_time.py [--out FILE] [--reps 100]

  - trainer.top_k_by_group over the 2,081,564 scores of the config-5 sweep (every RNA x protein pair of the
    NPInter2-shaped graph, RNA-major), grouped by RNA (4,636 groups of 449 pairs) and by protein (449 groups of 4,636),
    node serials as group ids (num_groups = 5,085 nodes), k = 10 and 100.  Scores: seeded uniform probabilities rounded
    to a 1e-4 grid, so that ties occur.  CUDA events over --reps calls after warm-up: the whole call (output and
    workspace allocation, the launches, its one synchronising read) one at a time, and npi_group_topk alone back to
    back into preallocated buffers.  Working set ~45 MB (scores, group ids, sort buffers), not flushed from the 126 MB
    L2 between calls.
  - the host route it replaces: device-to-host copy of the scores, then a stable numpy argsort of the [4,636, 449]
    score matrix along either axis, first k kept; checked equal to the GPU positions.
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
from npi_gnn_b200.trainer import top_k_by_group  # noqa: E402
from rank_time import device_info  # noqa: E402  (tools/rank_time.py, next to this script)


def events_ms(fn, reps):
    """(median, min) of one call at a time, and the mean of reps calls back to back."""
    per = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        e1.synchronize()
        per.append(e0.elapsed_time(e1))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return float(np.median(per)), float(np.min(per)), e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=100)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "topk_time.py measures on the GPU"
    torch.cuda.set_device(0)
    rec = {"tool": "tools/topk_time.py", **device_info()}
    d = synth.npinter2_shaped()
    allp = synth.all_candidate_pairs(d)
    V = len(d["is_rna"])
    R, P = int(d["is_rna"].sum()), int((d["is_rna"] == 0).sum())
    rng = np.random.default_rng(20240602)
    s_np = np.round(rng.random(len(allp)), 4).astype(np.float32)
    s = torch.as_tensor(s_np).cuda()
    rec.update(n=len(allp), num_groups=V, rna=R, protein=P)
    cases = {}
    for name, col in (("per_rna", 0), ("per_protein", 1)):
        grp = torch.as_tensor(allp[:, col].copy()).cuda()
        serials = np.nonzero(d["is_rna"] == (1 if col == 0 else 0))[0]
        for k in (10, 100):
            bufs = (torch.empty((V, k), dtype=torch.int32, device="cuda"), torch.empty((V, k), dtype=torch.float32, device="cuda"),
                    torch.empty(V, dtype=torch.int32, device="cuda"), torch.empty(1, dtype=torch.int32, device="cuda"),
                    torch.empty(ops.group_topk_workspace_bytes(len(allp), V), dtype=torch.uint8, device="cuda"))
            for _ in range(5):
                top_k_by_group(s, grp, V, k)
                ops.group_topk(s, grp, V, k, *bufs)
            torch.cuda.synchronize()
            call_med, call_min, _ = events_ms(lambda: top_k_by_group(s, grp, V, k), args.reps)
            raw_med, raw_min, raw_b2b = events_ms(lambda: ops.group_topk(s, grp, V, k, *bufs), args.reps)
            gpu_pos = top_k_by_group(s, grp, V, k)["pos"].cpu().numpy()[serials]
            host_ms = []
            for _ in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                m = s.cpu().numpy().reshape(R, P)
                if col == 0:
                    top = np.argsort(-m, axis=1, kind="stable")[:, :k] + (np.arange(R) * P)[:, None]
                else:
                    top = np.argsort(-m.T, axis=1, kind="stable")[:, :k] * P + np.arange(P)[:, None]
                host_ms.append((time.perf_counter() - t0) * 1e3)
            cases["%s_k%d" % (name, k)] = {
                "groups": len(serials), "members_per_group": len(allp) // len(serials), "k": k, "reps": args.reps,
                "top_k_by_group_ms_median": call_med, "top_k_by_group_ms_min": call_min,
                "group_topk_ms_median_isolated": raw_med, "group_topk_ms_min_isolated": raw_min,
                "group_topk_ms_back_to_back": raw_b2b,
                "numpy_argsort_host_ms_median": float(np.median(host_ms)), "numpy_argsort_host_ms_min": float(np.min(host_ms)),
                "equal_to_numpy": bool(np.array_equal(gpu_pos, top))}
    rec["top_k_by_group"] = cases
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
