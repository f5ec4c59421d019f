"""torchrun worker for the *_two_gpus_match_one tests of tests/test_gpu_rank.py, test_gpu_topk.py and
test_gpu_partner_rank.py: Scorer(world_size=2).<method>() on the NPInter2 fold-0 test set gives the same, bit-identical
result on both ranks, equal to the single-GPU result.  <method> (the argument): rank_metrics, top_partners or
partner_ranks; partner_ranks also scores the candidate pairs of 30 RNAs."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from npi_gnn_b200 import dist as D  # noqa: E402
from npi_gnn_b200.engine import FlatParams  # noqa: E402
from npi_gnn_b200.graph import BipartiteGraph, PairSet  # noqa: E402
from npi_gnn_b200.trainer import Scorer  # noqa: E402
from tests.common import load_ckpt, load_npinter2  # noqa: E402


def _rank0(t):
    """Rank 0's copy of ``t``."""
    other = t.clone()
    torch.distributed.broadcast(other, src=0)
    return other


def rank_metrics(dp, one, rank, world, dev):
    for k in ("auroc", "ap", "pr_auc_trapz", "n_pos", "n_neg", "twice_u", "confusion"):
        assert dp[k] == one[k], (rank, k, dp[k], one[k])
    for k in ("thresholds", "fpr", "tpr", "precision", "recall"):
        assert torch.equal(dp[k], one[k]), (rank, k)
        assert torch.equal(_rank0(dp[k]), dp[k]), (rank, k)
    row = torch.tensor([dp["auroc"], dp["ap"], dp["pr_auc_trapz"], float(dp["twice_u"])], dtype=torch.float64, device=dev)
    rows = D.gather_rows(row, dev)
    assert torch.equal(rows[0], rows[1])
    return ("RANK_DP world=%d auroc=%.12f ap=%.12f pr_auc_trapz=%.12f" % (world, dp["auroc"], dp["ap"], dp["pr_auc_trapz"]),
            "RANK_DP_OK")


def top_partners(dp, one, rank, world, dev):
    for side in ("rna", "protein"):
        for key in ("partner", "prob", "count"):
            a, b = dp[side][key], one[side][key]
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (rank, side, key)
            assert torch.equal(_rank0(a).view(torch.int32), a.view(torch.int32)), (rank, side, key)
    return ("TOPK_DP world=%d rna rows=%d protein rows=%d" % (world, int((dp["rna"]["count"] > 0).sum()),
                                                             int((dp["protein"]["count"] > 0).sum())),
            "TOPK_DP_OK")


def partner_ranks(dp, one, rank, world, dev):
    for side in ("rna", "protein"):
        for key in ("mrr", "hits", "n_queries", "n_unranked", "n_groups_scored"):
            assert dp[side][key] == one[side][key], (rank, side, key)
        assert np.float64(dp[side]["auc_macro"]).view(np.int64) == np.float64(one[side]["auc_macro"]).view(np.int64)
        for key in ("n_pos", "n_neg", "twice_u", "auc"):
            a, b = dp[side][key], one[side][key]
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (rank, side, key)
            assert torch.equal(_rank0(a).view(torch.int32), a.view(torch.int32)), (rank, side, key)
        summary = torch.tensor([dp[side]["mrr"], dp[side]["auc_macro"]], dtype=torch.float64, device=dev)
        assert torch.equal(_rank0(summary).view(torch.int64), summary.view(torch.int64)), (rank, side)
    return ("PARTNER_RANK_DP world=%d rna MRR %.5f (%d queries), protein MRR %.5f (%d queries)"
            % (world, dp["rna"]["mrr"], dp["rna"]["n_queries"], dp["protein"]["mrr"], dp["protein"]["n_queries"]),
            "PARTNER_RANK_DP_OK")


# method -> (call on a Scorer, comparison of the sharded and the single-GPU result)
METHODS = {
    "rank_metrics": (lambda sc: sc.rank_metrics(curve=True), rank_metrics),
    "top_partners": (lambda sc: sc.top_partners(20), top_partners),
    "partner_ranks": (lambda sc: sc.partner_ranks(), partner_ranks),
}


def main():
    method = sys.argv[1]
    run, compare = METHODS[method]
    world, rank, local = D.init("nccl")
    dev = torch.device("cuda", local)
    d = load_npinter2()
    g = BipartiteGraph(d["edges"], d["is_rna"], d["table"], device=dev)
    g.set_mask(np.concatenate([d["test_pos"], d["test_neg"]]))
    pairs = np.concatenate([d["test_pos"], d["test_neg"]])
    ys = np.concatenate([np.ones(len(d["test_pos"])), np.zeros(len(d["test_neg"]))]).astype(np.int32)
    if method == "partner_ranks":
        cand = g.candidate_pairs()
        cand = cand[np.isin(cand[:, 0], np.unique(d["test_pos"][:, 0])[:30])]
        pairs = np.concatenate([pairs, cand])
        ys = np.concatenate([ys, np.zeros(len(cand), dtype=np.int32)])
    perm = np.random.default_rng(0).permutation(len(pairs))
    ps = PairSet(g, pairs[perm], ys[perm], h=1)
    params = FlatParams(g.F, dev).load_state_dict(load_ckpt("ckpt_1223_1_15.npz"))
    dp = run(Scorer(ps, params, batch_size=200, world_size=world, rank=rank))
    one = run(Scorer(ps, params, batch_size=200))
    lines = compare(dp, one, rank, world, dev)
    D.barrier()
    if rank == 0:
        print("\n".join(lines))


if __name__ == "__main__":
    main()
