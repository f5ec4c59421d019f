"""Time Explainer.explain on the GPU and write one JSON record (device name and power limit read in the same run).

    python tools/explain_time.py [--out FILE] [--reps 3] [--host-pairs 400]

Two workloads, each explained with target 1, wrt "logp", full=False, 200 pairs per batch:
  - npinter2_test: the 4,166 NPInter2 fold-0 test pairs (2,083 positive + 2,083 negative) at h = 2 with the shipped
    checkpoint ckpt_1223_1_5 (the case the explanation of a held-out prediction serves).
  - config5_top10: the top-10 partners of every RNA of the config-5 sweep -- every RNA x protein pair of the
    NPInter2-shaped synthetic graph (2,081,564 pairs) scored by Scorer at h = 2 with the same checkpoint, then
    Scorer.top_partners(10)["rna"] -- about 46 k pairs (the sweep itself is not timed).
Per workload:
  - explain() from the call to its return (it ends in a synchronising read), CUDA events, median and min of --reps runs
    after one warm-up run;
  - the share of npi_input_attribution: one more run with CUDA events around every attribution call (events only, no
    synchronisation inside the sweep), their sum over that run's total;
  - Explainer.top_nodes(result, 10);
  - the host route it replaces: the fp32 oracle (oracle/net.py) under autograd on the CPU, batches of 200 collated on
    the host (oracle/khop_cwrap.py), x.requires_grad_(), logp[:, 1].sum().backward(), on the first --host-pairs pairs
    (pairs/s; the host route is timed on a prefix because it takes minutes per thousand pairs).
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from npi_gnn_b200 import _lib as L, synth  # noqa: E402
from npi_gnn_b200.engine import FlatParams  # noqa: E402
from npi_gnn_b200.graph import BipartiteGraph, PairSet  # noqa: E402
from npi_gnn_b200.trainer import Explainer, Scorer  # noqa: E402
from oracle import khop, khop_cwrap, net as onet  # noqa: E402
from rank_time import device_info  # noqa: E402  (tools/rank_time.py, next to this script)
from tests.common import load_ckpt, load_npinter2  # noqa: E402

CKPT = "ckpt_1223_1_5.npz"
B = 200


class AttributionEvents:
    """L.TIMER: CUDA events around every npi_input_attribution call."""

    def __init__(self):
        self.pairs = []

    def begin(self, name):
        if name == "npi_input_attribution":
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self.pairs.append([e, None])

    def end(self, name):
        if name == "npi_input_attribution":
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self.pairs[-1][1] = e

    def total_ms(self):
        return sum(a.elapsed_time(b) for a, b in self.pairs)


def timed_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def host_route(pairs, ys, h, table, og, omask, sd, F):
    m = onet.Net_1(F)
    m.load_state_dict(sd)
    m.eval()
    t0 = time.perf_counter()
    for i in range(0, len(pairs), B):
        c = khop_cwrap.collate_batch(og, omask, pairs[i:i + B], ys[i:i + B], h, table)
        bn = onet.batch_namespace(c)
        x = bn.x.float().requires_grad_()
        bn.x = x
        m(bn)[:, 1].sum().backward()
        (x.detach() * x.grad).sum(1)
    return time.perf_counter() - t0


def workload(ps, params, pairs, ys, table, og, omask, sd, args):
    ex = Explainer(ps, params, batch_size=B)
    ex.explain()                                                    # warm-up
    torch.cuda.synchronize()
    ms = [timed_ms(ex.explain)[0] for _ in range(args.reps)]
    ev = AttributionEvents()
    L.TIMER = ev
    try:
        total, res = timed_ms(ex.explain)
    finally:
        L.TIMER = None
    attrib = ev.total_ms()
    Explainer.top_nodes(res, 10)
    top_ms = timed_ms(lambda: Explainer.top_nodes(res, 10))[0]
    P = len(pairs)
    nh = min(args.host_pairs, P)
    host_s = host_route(pairs[:nh], ys[:nh], 2, table, og, omask, sd, ps.graph.F)
    return {"pairs": P, "rows": int(ps.n_h.sum()), "batches": (P + B - 1) // B, "tiny_path": bool(ex.engine.tiny),
            "explain_ms_median": float(np.median(ms)), "explain_ms_min": float(np.min(ms)),
            "pairs_per_s": P / (float(np.median(ms)) / 1e3),
            "attribution_ms": attrib, "attribution_calls": len(ev.pairs), "attribution_share": attrib / total,
            "top_nodes10_ms": top_ms,
            "host_fp32_oracle_pairs": nh, "host_fp32_oracle_s": host_s, "host_fp32_oracle_pairs_per_s": nh / host_s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-pairs", type=int, default=400)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "explain_time.py measures on the GPU"
    torch.cuda.set_device(0)
    torch.set_num_threads(os.cpu_count() or 1)
    rec = {"tool": "tools/explain_time.py", **device_info(), "batch": B, "checkpoint": CKPT, "cpu_threads": torch.get_num_threads()}
    sd = load_ckpt(CKPT)

    d = load_npinter2()
    test = np.concatenate([d["test_pos"], d["test_neg"]])
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device="cuda")
    g.set_mask(test)
    og = khop.build_csr([tuple(e) for e in d["edges"].tolist()], d["is_rna"])
    omask = khop.mask_from_keys(og, [tuple(e) for e in test.tolist()])
    ys = np.concatenate([np.ones(len(d["test_pos"])), np.zeros(len(d["test_neg"]))]).astype(np.int32)
    params = FlatParams(g.F, "cuda").load_state_dict(sd)
    rec["npinter2_test"] = workload(PairSet(g, test, ys, h=2), params, test, ys, d["table"], og, omask, sd, args)
    print(json.dumps(rec["npinter2_test"]), flush=True)

    s = synth.npinter2_shaped()
    cannot = synth.masked_pairs(s)
    g5 = BipartiteGraph(s["edges"], s["is_rna"], s["table"], device="cuda")
    g5.set_mask(cannot)
    allp = synth.all_candidate_pairs(s)
    params5 = FlatParams(g5.F, "cuda").load_state_dict(sd)
    top = Scorer(PairSet(g5, allp, np.zeros(len(allp), dtype=np.int32), h=2), params5, batch_size=2048).top_partners(10)["rna"]
    partner, count = top["partner"].cpu().numpy(), top["count"].cpu().numpy()
    rna = np.nonzero(count > 0)[0]
    pairs5 = np.stack([np.repeat(rna, count[rna]), np.concatenate([partner[r, :count[r]] for r in rna])], 1).astype(np.int32)
    ys5 = np.zeros(len(pairs5), dtype=np.int32)
    og5 = khop.build_csr([tuple(e) for e in s["edges"].tolist()], s["is_rna"])
    omask5 = khop.mask_from_keys(og5, [tuple(e) for e in cannot.tolist()])
    rec["config5_top10"] = workload(PairSet(g5, pairs5, ys5, h=2), params5, pairs5, ys5, s["table"], og5, omask5,
                                    sd, args)
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
